// Exercises the volume source of the C++ wrapper (wave-fenics_b200/hpp/wavefx.hpp): a LossyGLLOpt in a
// wavefx::Medium with a layer and set_volume_source, 15 steps, a checkpoint of u, v, psi and phi fed back through
// set_state and set_pml_state, 15 more steps.  The mesh, weights, layer, source and initial state come from raw fp64 /
// int32 files written by tests/test_volume_source.py (argv[1] names their directory); the final u is written back
// there for a bitwise comparison with the Python model.  Prints "volume source hpp ok".  Needs a GPU to run, only a
// compiler to build.
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

template <typename F>
static bool refused(F&& f)
{
  try
  {
    f();
  }
  catch (const std::runtime_error&)
  {
    return true;
  }
  return false;
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
    // params: P, c0, f0, p0, delta, dt
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
    wavefx::PML pml;
    pml.zeta = load<double>(dir, "zeta.f64");
    const int P = (int)par[0];
    const double c0 = par[1], f0 = par[2], p0 = par[3], delta = par[4], dt = par[5];
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
    wavefx::LossyGLLOpt lossy(ctx, V, P, c0, f0, p0, delta, med);
    lossy.set_pml(V, pml);
    lossy.set_volume_source(load<std::int32_t>(dir, "sdofs.i32"), load<double>(dir, "sq.f64"),
                            load<double>(dir, "sdelay.f64"));
    lossy.set_state(u0, v0);
    auto steps = [&](double t0) {
      std::int64_t n = 0;
      double t = 0;
      wavefx::check(wfx_wave_rk4(lossy.get(), t0, 1.0, dt, 15, &n, &t, nullptr));
      if (n != 15) throw std::runtime_error("expected 15 steps");
      return t;
    };
    const double t1 = steps(0.0);
    std::vector<double> u, v, psi, phi;
    lossy.solution(u, v);
    lossy.pml_state(psi, phi);
    lossy.set_state(u, v);
    lossy.set_pml_state(psi, phi);
    steps(t1);
    lossy.solution(u, v);
    lossy.pml_state(psi, phi);
    save(dir, "u.out.f64", u);
    // short weights, a duplicate dof and a negative delay are refused
    const std::vector<std::int32_t> two = {3, 5}, dup = {3, 3};
    if (!refused([&] { lossy.set_volume_source(two, {1.0}, {}); }))
      throw std::runtime_error("short weights were accepted");
    if (!refused([&] { lossy.set_volume_source(dup, {1.0, 1.0}, {}); }))
      throw std::runtime_error("a duplicate dof was accepted");
    if (!refused([&] { lossy.set_volume_source(two, {1.0, 1.0}, {0.0, -1e-6}); }))
      throw std::runtime_error("a negative delay was accepted");
  }
  catch (const std::exception& e)
  {
    std::fprintf(stderr, "volume source hpp FAILED: %s\n", e.what());
    return 1;
  }
  std::printf("volume source hpp ok\n");
  return 0;
}
