// Exercises the layered-medium constructors of the C++ wrapper (wave-fenics_b200/hpp/wavefx.hpp): LinearGLLOpt,
// LossyGLLOpt, WesterveltGLLOpt and LinearGLLEnsemble with a wavefx::Medium.  The mesh, the medium's weights and the
// initial state come from raw fp64 / int32 files written by tests/test_media.py (argv[1] names their directory); each
// model's final u is written back there for a bitwise comparison with the Python models.  Prints "medium hpp ok".
// Needs a GPU to run, only a compiler to build.
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
    // params: P, c0, f0, p0, delta, beta, rho0, t0, tf, dt
    const auto par = load<double>(dir, "params.f64");
    const auto x = load<double>(dir, "x.f64");
    const auto xdofs = load<std::int32_t>(dir, "xdofs.i32");
    const auto dofmap = load<std::int32_t>(dir, "dofmap.i32");
    const auto fcell = load<std::int32_t>(dir, "fcell.i32"), flocal = load<std::int32_t>(dir, "flocal.i32"),
               ftag = load<std::int32_t>(dir, "ftag.i32");
    const auto u0 = load<double>(dir, "u.f64"), v0 = load<double>(dir, "v.f64");
    wavefx::Medium med;
    med.stiffness = load<double>(dir, "stiffness.f64");
    med.mass = load<double>(dir, "mass.f64");
    med.facet = load<double>(dir, "facet.f64");
    med.kappa = load<double>(dir, "kappa.f64");
    const int P = (int)par[0];
    const double c0 = par[1], f0 = par[2], p0 = par[3], delta = par[4], beta = par[5], rho0 = par[6];
    double t0 = par[7], tf = par[8], dt = par[9];
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
    std::vector<double> u, v;
    auto run = [&](wavefx::LinearGLLOpt& m, const char* out) {
      m.set_state(u0, v0);
      double a = t0, b = tf, h = dt;
      m.rk4(a, b, h);
      m.solution(u, v);
      save(dir, out, u);
    };
    wavefx::Medium lin = med;
    lin.kappa.clear();
    wavefx::LinearGLLOpt linear(ctx, V, P, c0, f0, p0, lin);
    run(linear, "u_linear.f64");
    wavefx::LossyGLLOpt lossy(ctx, V, P, c0, f0, p0, delta, lin);
    run(lossy, "u_lossy.f64");
    wavefx::WesterveltGLLOpt west(ctx, V, P, c0, f0, p0, delta, beta, rho0, med);
    run(west, "u_westervelt.f64");
    // two members, both the state of the single-field runs, member 0 with (f0, p0)
    wavefx::LinearGLLEnsemble ens(ctx, V, P, c0, {f0, 0.7 * f0}, {p0, 0.5 * p0}, lin);
    std::vector<double> U(2 * u0.size()), W(2 * u0.size());
    for (std::size_t i = 0; i < u0.size(); ++i)
    {
      U[2 * i] = U[2 * i + 1] = u0[i];
      W[2 * i] = W[2 * i + 1] = v0[i];
    }
    ens.set_state(U, W);
    double a = t0, b = tf, h = dt;
    ens.rk4(a, b, h);
    ens.solution(U, W);
    save(dir, "u_ensemble.f64", U);
    // a medium with the wrong number of weights is refused
    wavefx::Medium bad = lin;
    bad.mass.pop_back();
    bool refused = false;
    try
    {
      wavefx::LinearGLLOpt m(ctx, V, P, c0, f0, p0, bad);
    }
    catch (const std::runtime_error&)
    {
      refused = true;
    }
    if (!refused) throw std::runtime_error("a short medium was accepted");
  }
  catch (const std::exception& e)
  {
    std::fprintf(stderr, "medium hpp FAILED: %s\n", e.what());
    return 1;
  }
  std::printf("medium hpp ok\n");
  return 0;
}
