// wavefx.hpp -- header-only C++17 wrappers over the C ABI (include/wavefx.h) with the call
// shape of the reference classes, so that host code written against
//   common/operators.hpp   MassOperatorCPU<T>(V, degree), StiffnessOperator<T>(V, degree, params),
//                          void operator()(const Vector& x, Vector& y)   ==>  y += A x
//   common/LinearGLL.hpp   LinearGLLOpt(mesh, meshtags, degree, c0, f0, p0), init(), rk4(t0, tf, dt)
// can switch to the B200 path by changing the include and the type of `V`.
//
// The reference pulls everything it needs out of a dolfinx::fem::FunctionSpace.  DOLFINx is not
// a dependency here: `wavefx::SpaceView` carries the same arrays as plain pointers, and
// INTEGRATION.md shows the six-line adapter that fills it from a FunctionSpace.
// Vectors are any type with data() and size() over contiguous T (std::vector<T>,
// dolfinx::la::Vector<T>::mutable_array(), xtl::span<T>) holding HOST memory in DOLFINx layout
// [owned | ghosts]; the *_device overloads take raw device pointers and a cudaStream_t.
// Errors become std::runtime_error like the reference's CUDA classes
// (common/cuda/array.hpp:15-17).
#pragma once

#include "wavefx.h"

#include <array>
#include <complex>
#include <cstdint>
#include <functional>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <vector>

namespace wavefx
{
inline void check(int status)
{
  if (status != 0) throw std::runtime_error(std::string("wavefx: ") + wfx_last_error());
}

template <typename T>
constexpr int dtype_of()
{
  static_assert(std::is_same_v<T, double> || std::is_same_v<T, float>, "T must be double or float");
  return std::is_same_v<T, double> ? WFX_F64 : WFX_F32;
}

// What the operators read from V (fem::FunctionSpace) and its mesh.
struct SpaceView
{
  int degree = 0;
  std::int64_t ncells = 0;               // mesh->topology().index_map(tdim)->size_local()
  std::int64_t npoints = 0;              // geometry.x().size() / 3
  const double* x = nullptr;             // geometry.x().data()
  const std::int32_t* xdofs = nullptr;   // geometry.dofmap().array().data()  [ncells][8]
  std::int64_t ndofs = 0;                // index_map->size_local() + num_ghosts()
  std::int64_t size_local = 0;           // index_map->size_local()
  const std::int32_t* dofmap = nullptr;  // V->dofmap()->list().array().data()  [ncells][(P+1)^3]
  // exterior facets with tags (the MeshTags handed to create_form, LinearGLL.hpp:113-115)
  std::int64_t nfacets = 0;
  const std::int32_t* facet_cell = nullptr;
  const std::int32_t* facet_local = nullptr;
  const std::int32_t* facet_tag = nullptr;
};

class Context
{
public:
  explicit Context(int device = 0) { check(wfx_ctx_create(device, &_h)); }
  ~Context() { wfx_ctx_destroy(_h); }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;
  wfx_ctx* get() const { return _h; }
  void synchronize() const { check(wfx_ctx_sync(_h)); }

private:
  wfx_ctx* _h = nullptr;
};

// precompute_geometric_data(mesh, p) (common/precomputation.hpp:18-110)
template <typename T>
class Geometry
{
public:
  Geometry(std::shared_ptr<Context> ctx, const SpaceView& V) : _ctx(std::move(ctx))
  {
    check(wfx_geometry_create(_ctx->get(), V.degree, dtype_of<T>(), V.ncells, V.npoints, V.x, V.xdofs, &_h));
  }
  ~Geometry() { wfx_geometry_destroy(_h); }
  Geometry(const Geometry&) = delete;
  Geometry& operator=(const Geometry&) = delete;
  wfx_geom* get() const { return _h; }
  const std::shared_ptr<Context>& context() const { return _ctx; }
  // (G [ncells][nq][3][3], detJ [ncells][nq]) in the reference layout
  void get(std::vector<double>& G, std::vector<double>& detJ, std::int64_t ncells, int nq) const
  {
    G.resize((std::size_t)ncells * nq * 9);
    detJ.resize((std::size_t)ncells * nq);
    check(wfx_geometry_get(_h, G.data(), detJ.data()));
  }
  // cells whose G is w_q times one constant matrix (parallelepipeds): all of them => the stiffness
  // operator takes the structured fast path (6 scalars of G per cell)
  std::int64_t num_affine_cells() const
  {
    std::int64_t nc = 0, na = 0;
    check(wfx_geometry_info(_h, &nc, &na));
    return na;
  }
  // heterogeneous medium: G of cell c scaled by coeff[c], e.g. (c0[c] / c0_ref)^2 -- the coefficient
  // the reference leaves as a TODO (common/LinearGLL.hpp:170, params ignored at operators.hpp:113-115)
  void scale_cells(const std::vector<double>& coeff) { check(wfx_geometry_scale_cells(_h, coeff.data())); }

private:
  std::shared_ptr<Context> _ctx;
  wfx_geom* _h = nullptr;
};

template <typename T>
class StiffnessOperator
{
public:
  // `params` is accepted and -- exactly like the reference (common/operators.hpp:113-115) --
  // not used for the speed of sound: c0 = 1500 is hard-coded there.
  // shared_dofs (distributed meshes): the local dofs that also live on another rank (the union of
  // HaloSpec::send_indices and recv_indices).  Cells touching them are scheduled first so that the
  // ghost exchange overlaps the interior cells.
  // flags: WFX_STIFF_ENSEMBLE adds the ensemble path (apply_ensemble_device)
  StiffnessOperator(std::shared_ptr<Geometry<T>> geom, const SpaceView& V, int bdegree,
                    std::map<std::string, double>& params, const std::vector<std::int32_t>& shared_dofs = {},
                    int flags = WFX_STIFF_AUTO)
      : _geom(std::move(geom)), _ndofs(V.ndofs), _params(params)
  {
    if (bdegree != V.degree) throw std::runtime_error("wavefx: degree mismatch");
    check(wfx_stiffness_create_partitioned(_geom->context()->get(), _geom->get(), V.ndofs, V.dofmap, 1500.0,
                                           flags, (std::int64_t)shared_dofs.size(),
                                           shared_dofs.empty() ? nullptr : shared_dofs.data(), &_h));
  }
  ~StiffnessOperator() { wfx_stiffness_destroy(_h); }
  StiffnessOperator(const StiffnessOperator&) = delete;
  StiffnessOperator& operator=(const StiffnessOperator&) = delete;

  // y += A x on host vectors (the reference functor, operators.hpp:182-200)
  template <typename VecIn, typename VecOut>
  void operator()(const VecIn& x, VecOut& y)
  {
    if ((std::int64_t)x.size() != _ndofs || (std::int64_t)y.size() != _ndofs)
      throw std::runtime_error("wavefx: vector size does not match the function space");
    check(wfx_stiffness_apply_host(_h, x.data(), y.data(), 1));
  }
  // device pointers, asynchronous on `stream`
  void apply_device(const T* x, T* y, int beta = 1, void* stream = nullptr)
  {
    check(wfx_stiffness_apply(_h, x, y, beta, stream));
  }
  void apply_scaled_device(const T* x, const T* scale, T* y, void* stream = nullptr)
  {
    check(wfx_stiffness_apply_scaled(_h, x, scale, y, stream));
  }
  // nv member-interleaved fields ([ndofs][nv], the blocked la::Vector with bs = nv) in one pass over G:
  // y[:,m] (+)= scale .* (-c0^2 K x[:,m]); scale (ndofs entries, e.g. 1/m) may be null and needs beta == 0
  void apply_ensemble_device(int nv, const T* x, const T* scale, T* y, int beta = 0, void* stream = nullptr)
  {
    check(wfx_stiffness_apply_ensemble(_h, nv, x, scale, y, beta, stream));
  }
  std::size_t num_cells() const { return (std::size_t)info().ncells; }
  std::size_t num_dofs() const { return (std::size_t)info().nd; }
  double flops() const { return info().flops; }
  // the structured fast path was selected (every cell affine, every batch a lattice brick)
  bool affine_fast_path() const
  {
    int variant = 0, affine = 0, mixed = 0, nreg = 0, nb = 0;
    std::int64_t smem = 0;
    check(wfx_stiffness_kernel_info(_h, &variant, &affine, &mixed, &nreg, &nb, &smem));
    return affine != 0;
  }
  wfx_stiffness* get() const { return _h; }

private:
  struct Info
  {
    std::int64_t ncells, ndofs;
    int nd, ncol, nl;
    double flops, bytes;
  };
  Info info() const
  {
    Info i{};
    check(wfx_stiffness_info(_h, &i.ncells, &i.nd, &i.ndofs, &i.flops, &i.bytes, &i.ncol, &i.nl));
    return i;
  }
  std::shared_ptr<Geometry<T>> _geom;
  std::int64_t _ndofs;
  std::map<std::string, double> _params;
  wfx_stiffness* _h = nullptr;
};

// MassOperatorCPU<T> (common/operators.hpp:43-109); LinearGLL.hpp:63 spells it MassOperator.
template <typename T>
class MassOperator
{
public:
  // cell_weight: one weight per cell (the weighted mass of a layered medium, DESIGN.md section 4.5e) or nullptr
  MassOperator(std::shared_ptr<Geometry<T>> geom, const SpaceView& V, int bdegree, const double* cell_weight = nullptr)
      : _geom(std::move(geom)), _ndofs(V.ndofs)
  {
    if (bdegree != V.degree) throw std::runtime_error("wavefx: degree mismatch");
    check(wfx_mass_create_weighted(_geom->context()->get(), _geom->get(), V.ndofs, V.dofmap, cell_weight, &_h));
  }
  ~MassOperator() { wfx_mass_destroy(_h); }
  MassOperator(const MassOperator&) = delete;
  MassOperator& operator=(const MassOperator&) = delete;
  template <typename VecIn, typename VecOut>
  void operator()(const VecIn& x, VecOut& y)
  {
    if ((std::int64_t)x.size() != _ndofs || (std::int64_t)y.size() != _ndofs)
      throw std::runtime_error("wavefx: vector size does not match the function space");
    check(wfx_mass_apply_host(_h, x.data(), y.data(), 1));
  }
  void apply_device(const T* x, T* y, int beta = 1, void* stream = nullptr) { check(wfx_mass_apply(_h, x, y, beta, stream)); }
  const T* inverse_diagonal_device() const
  {
    const void* p = nullptr;
    check(wfx_mass_inverse_diagonal(_h, &p));
    return static_cast<const T*>(p);
  }
  wfx_mass* get() const { return _h; }

private:
  std::shared_ptr<Geometry<T>> _geom;
  std::int64_t _ndofs;
  wfx_mass* _h = nullptr;
};
template <typename T>
using MassOperatorCPU = MassOperator<T>;

// y_i = M^-1 (-c0^2 K x_i) for several HOST vectors in one call: copy-in, fused apply and copy-out of
// consecutive vectors are pipelined (use pinned memory), see wfx_stiffness_mass_apply_host_batch.
template <typename T>
void stiffness_mass_apply_batch(StiffnessOperator<T>& K, MassOperator<T>& M, const std::vector<const T*>& x,
                                const std::vector<T*>& y)
{
  if (x.size() != y.size()) throw std::runtime_error("wavefx: x and y lists differ in length");
  check(wfx_stiffness_mass_apply_host_batch(K.get(), M.get(), (int)x.size(), reinterpret_cast<const void* const*>(x.data()),
                                            reinterpret_cast<void* const*>(y.data())));
}

// Index data of a ghost exchange, as VectorUpdater reads it from the IndexMap
// (demo/gpu_scatter_mpi/VectorUpdater.hpp:31-59 and the neighbour ranks of :69-80).
struct HaloSpec
{
  std::vector<std::int32_t> send_ranks;   // destination ranks of the forward scatter
  std::vector<std::int32_t> send_offsets; // scatter_fwd_indices().offsets()
  std::vector<std::int32_t> send_indices; // scatter_fwd_indices().array(): owned local indices
  std::vector<std::int32_t> recv_ranks;   // source ranks of the forward scatter
  std::vector<std::int32_t> recv_offsets; // scatter_fwd_receive_offsets()
  std::vector<std::int32_t> recv_indices; // size_local + scatter_fwd_ghost_positions()[i]: local ghost slots
  std::int64_t size_local = 0;            // index_map->size_local()
  std::int64_t num_ghosts = 0;            // index_map->num_ghosts()
};

// The NCCL communicator that takes the place of the IndexMap's MPI neighbourhood communicators.
// `id` comes from Comm::unique_id() on rank 0 and is distributed by the caller
// (MPI_Bcast(id.data(), 128, MPI_BYTE, 0, comm)).
class Comm
{
public:
  static std::array<char, 128> unique_id()
  {
    std::array<char, 128> id{};
    check(wfx_comm_unique_id(id.data()));
    return id;
  }
  Comm(std::shared_ptr<Context> ctx, const std::array<char, 128>& id, int nranks, int rank) : _ctx(std::move(ctx))
  {
    check(wfx_comm_create(_ctx->get(), id.data(), nranks, rank, &_h));
  }
  ~Comm() { wfx_comm_destroy(_h); }
  Comm(const Comm&) = delete;
  Comm& operator=(const Comm&) = delete;
  wfx_comm* get() const { return _h; }
  const std::shared_ptr<Context>& context() const { return _ctx; }

private:
  std::shared_ptr<Context> _ctx;
  wfx_comm* _h = nullptr;
};

// VectorUpdater<T> (demo/gpu_scatter_mpi/VectorUpdater.hpp:21-215): owner -> ghost copy and
// ghost -> owner add on DEVICE arrays laid out [owned | ghosts].  The begin/end pairs of the
// reference collapse to one asynchronous call on the given stream.
template <typename T>
class VectorUpdater
{
public:
  VectorUpdater(std::shared_ptr<Comm> comm, const HaloSpec& s) : _comm(std::move(comm))
  {
    check(wfx_halo_create(_comm->context()->get(), _comm->get(), std::is_same<T, double>::value ? WFX_F64 : WFX_F32,
                          s.size_local, s.num_ghosts, (int)s.send_ranks.size(), s.send_ranks.data(), s.send_offsets.data(), s.send_indices.data(),
                          (int)s.recv_ranks.size(), s.recv_ranks.data(), s.recv_offsets.data(), s.recv_indices.data(),
                          &_h));
  }
  ~VectorUpdater() { wfx_halo_destroy(_h); }
  VectorUpdater(const VectorUpdater&) = delete;
  VectorUpdater& operator=(const VectorUpdater&) = delete;
  void update_fwd(T* x_dev, void* stream = nullptr) { check(wfx_halo_update_fwd(_h, x_dev, stream)); }          // :148
  void update_rev(T* x_dev, void* stream = nullptr) { check(wfx_halo_update_rev(_h, x_dev, stream)); }          // :204
  // reverse add then forward copy in one call: every copy of a shared dof ends bitwise identical
  void update_rev_fwd(T* x_dev, void* stream = nullptr) { check(wfx_halo_update_rev_fwd(_h, x_dev, stream)); }
  wfx_halo* get() const { return _h; }

private:
  std::shared_ptr<Comm> _comm;
  wfx_halo* _h = nullptr;
};

// Field statistics of a wave model (wfx_wave_set_field_stats, DESIGN.md section 4.5b), host copies: N sampled
// steps from t_first to t_last, peaks shaped like the state, harmonics[(h - 1) * entries + i] the amplitude
// (2 / N) sum_n u_i(t_n) exp(-i h w t_n) of harmonic h at state entry i.
struct FieldStats
{
  std::int64_t samples = 0;
  double t_first = 0, t_last = 0;
  std::vector<double> pmax, pmin;
  std::vector<std::complex<double>> harmonics;
};
inline void read_field_stats(wfx_wave* wave, std::int64_t entries, FieldStats& out)
{
  int enabled = 0, nharm = 0; // the library's own setting sizes the buffers
  check(wfx_wave_field_stats_info(wave, &enabled, nullptr, &nharm));
  if (!enabled) throw std::runtime_error("wavefx: field statistics are off (set_field_stats)");
  out.pmax.resize((std::size_t)entries);
  out.pmin.resize((std::size_t)entries);
  out.harmonics.resize((std::size_t)(entries * nharm));
  check(wfx_wave_get_field_stats(wave, &out.samples, &out.t_first, &out.t_last, out.pmax.data(), out.pmin.data(),
                                 reinterpret_cast<double*>(out.harmonics.data())));
}
// wfx_wave_set_source_profile over `entries` state entries; an empty vector is passed as NULL
inline void set_profile(wfx_wave* wave, std::int64_t entries, const std::vector<double>& amp,
                        const std::vector<double>& delay)
{
  for (const auto* a : {&amp, &delay})
    if (!a->empty() && (std::int64_t)a->size() != entries)
      throw std::runtime_error("wavefx: source profile arrays must hold one entry per state entry (or none)");
  check(wfx_wave_set_source_profile(wave, amp.empty() ? nullptr : amp.data(), delay.empty() ? nullptr : delay.data()));
}
// wfx_wave_set_volume_source with nv weights / delays per dof; an empty delay vector is passed as NULL
inline void set_volume(wfx_wave* wave, int nv, const std::vector<std::int32_t>& dofs, const std::vector<double>& q,
                       const std::vector<double>& delay)
{
  const std::size_t ne = dofs.size() * (std::size_t)nv;
  if (q.size() != ne || (!delay.empty() && delay.size() != ne))
    throw std::runtime_error("wavefx: volume source weights and delays must hold nv entries per dof");
  check(wfx_wave_set_volume_source(wave, (std::int64_t)dofs.size(), dofs.data(), q.data(),
                                   delay.empty() ? nullptr : delay.data()));
}

// A layered medium (DESIGN.md section 4.5e) as the weights of the operators, e.g. from the Python Medium class:
//   stiffness [ncells]  rho_ref / rho_c                         (scales the model's geometry)
//   mass      [ncells]  rho_ref c0^2 / (rho_c c_c^2)            (weighted lumped mass)
//   facet     [nfacets] rho_ref / rho_f on tag 1, rho_ref c0 / (rho_f c_f) on tag 2, 1 elsewhere
//   kappa     [ndofs]   the per-dof nonlinearity of the Westervelt model; empty: the model's scalar kappa
struct Medium
{
  std::vector<double> stiffness, mass, facet, kappa;
};
inline void check_medium(const SpaceView& V, const Medium& m)
{
  if ((std::int64_t)m.stiffness.size() != V.ncells || (std::int64_t)m.mass.size() != V.ncells ||
      (std::int64_t)m.facet.size() != V.nfacets)
    throw std::runtime_error("wavefx: medium needs stiffness and mass weights per cell and a weight per facet");
}

// A perfectly matched layer (DESIGN.md section 4.5g) as its damping profile, e.g. the Python PML.zeta:
//   zeta [3][ndofs]  >= 0 [1/s] along physical axis j; the layer is the cells where some zeta_j > 0 at a point
struct PML
{
  std::vector<double> zeta;
};

// The wave model and its RK4 driver (common/LinearGLL.hpp:37-287), fp64 like the reference.
class LinearGLLOpt
{
public:
  // halo: the fp64 ghost exchange of a distributed mesh (nullptr on one rank); it must outlive the model
  LinearGLLOpt(std::shared_ptr<Context> ctx, const SpaceView& V, int& degreeOfBasis, double& speedOfSound,
               double& sourceFrequency, double& pressureAmplitude,
               std::shared_ptr<VectorUpdater<double>> halo = nullptr, const HaloSpec* spec = nullptr)
      : _ctx(std::move(ctx)), _halo(std::move(halo)), _ndofs(V.ndofs), _nq((std::int64_t)(V.degree + 1) * (V.degree + 1) * (V.degree + 1))
  {
    std::vector<std::int32_t> shared;
    if (spec)
    {
      shared = spec->send_indices;
      shared.insert(shared.end(), spec->recv_indices.begin(), spec->recv_indices.end());
    }
    _geom = std::make_shared<Geometry<double>>(_ctx, V);
    mass_op = std::make_shared<MassOperator<double>>(_geom, V, degreeOfBasis);                 // :105
    std::map<std::string, double> params{{"c0", speedOfSound}};
    stiff_op = std::make_shared<StiffnessOperator<double>>(_geom, V, degreeOfBasis, params, shared);  // :120
    check(wfx_boundary_create(_ctx->get(), V.degree, WFX_F64, V.nfacets, V.facet_cell, V.facet_local,
                              V.facet_tag, V.npoints, V.x, V.xdofs, V.ndofs, V.dofmap, &_bnd));  // :113-115
    check(wfx_wave_create(_ctx->get(), stiff_op->get(), mass_op->get(), _bnd, _halo ? _halo->get() : nullptr, V.size_local,
                          speedOfSound, sourceFrequency, pressureAmplitude, &_wave));
  }
  // the same model in a layered medium (one rank)
  LinearGLLOpt(std::shared_ptr<Context> ctx, const SpaceView& V, int degreeOfBasis, double speedOfSound,
               double sourceFrequency, double pressureAmplitude, const Medium& medium)
      : _ctx(std::move(ctx)), _ndofs(V.ndofs), _nq((std::int64_t)(V.degree + 1) * (V.degree + 1) * (V.degree + 1))
  {
    make_operators(V, degreeOfBasis, speedOfSound, &medium);
    check(wfx_wave_create(_ctx->get(), stiff_op->get(), mass_op->get(), _bnd, nullptr, V.size_local, speedOfSound,
                          sourceFrequency, pressureAmplitude, &_wave));
  }
  ~LinearGLLOpt()
  {
    wfx_wave_destroy(_wave);
    wfx_pml_destroy(_pml);
    wfx_boundary_destroy(_bnd);
  }
  LinearGLLOpt(const LinearGLLOpt&) = delete;
  LinearGLLOpt& operator=(const LinearGLLOpt&) = delete;

  void init() { check(wfx_wave_init(_wave)); }                                                  // :131-134
  // the right-hand sides on their own (:141-192), device arrays of ndofs entries
  void f0(double t, const double* u_dev, const double* v_dev, double* result_dev, void* stream = nullptr)
  {
    check(wfx_wave_f0(_wave, t, u_dev, v_dev, result_dev, stream));
  }
  void f1(double t, const double* u_dev, const double* v_dev, double* result_dev, void* stream = nullptr)
  {
    check(wfx_wave_f1(_wave, t, u_dev, v_dev, result_dev, stream));
  }
  // rk4(startTime, finalTime, timeStep) (:198-287); returns the number of steps taken
  std::int64_t rk4(double& startTime, double& finalTime, double& timeStep)
  {
    std::int64_t steps = 0;
    double t_end = 0;
    check(wfx_wave_rk4(_wave, startTime, finalTime, timeStep, 0, &steps, &t_end, nullptr));
    _ctx->synchronize();
    return steps;
  }
  // ---- output (the reference prints the solve time only, demo/cpu_planar3d/main.cpp:87-93) ----
  // u at the given dofs after every completed step, kept on the device (at most max_records steps)
  void set_probes(const std::vector<std::int32_t>& dofs, std::int64_t max_records)
  {
    _nprobes = (std::int64_t)dofs.size();
    check(wfx_wave_set_probes(_wave, _nprobes, dofs.data(), max_records));
  }
  // times [nrec] and values [nrec][nprobes] recorded so far
  void probe_series(std::vector<double>& t, std::vector<double>& values) const
  {
    std::int64_t n = 0;
    check(wfx_wave_get_probe_series(_wave, &n, nullptr, nullptr));
    t.resize((std::size_t)n);
    values.resize((std::size_t)(n * _nprobes));
    check(wfx_wave_get_probe_series(_wave, &n, t.data(), values.data()));
  }
  // peaks and harmonics 1..nharm (<= WFX_HARMONICS_MAX) of u over the steps with t_n >= t_start - dt/2, kept on
  // the device; resets them (so do init and set_state).  enable = false switches them off.
  void set_field_stats(bool enable, double t_start = 0.0, int nharm = 0)
  {
    check(wfx_wave_set_field_stats(_wave, enable ? 1 : 0, t_start, nharm));
  }
  void field_stats(FieldStats& out) const { read_field_stats(_wave, _ndofs, out); }
  // phased-array source on tag 1 (DESIGN.md section 4.5c): amp[i] g(t - delay[i]) in place of g(t), ndofs entries
  // each; an empty vector stands for amp = 1 / delay = 0, both empty clear the profile
  void set_source_profile(const std::vector<double>& amp, const std::vector<double>& delay)
  {
    set_profile(_wave, _ndofs, amp, delay);
  }
  // volume source (DESIGN.md section 4.5h): c0^2 q[p] g(t - delay[p]) added at dof dofs[p] (distinct dofs; an empty
  // delay stands for 0, empty dofs clear the source); a point source's weights are the basis functions at the point
  void set_volume_source(const std::vector<std::int32_t>& dofs, const std::vector<double>& q,
                         const std::vector<double>& delay)
  {
    set_volume(_wave, 1, dofs, q, delay);
  }
  // fn(step, t, u, v) every `every` steps with pointers into pinned host copies (ndofs entries each);
  // the device -> host copy overlaps the time stepping.  A checkpoint is a snapshot handed back to
  // set_state.
  void set_snapshot(std::int64_t every, std::function<void(std::int64_t, double, const double*, const double*)> fn)
  {
    _snap = std::move(fn);
    check(wfx_wave_set_snapshot(_wave, _snap ? every : 0, _snap ? &LinearGLLOpt::snapshot_trampoline : nullptr, this));
  }
  void set_state(const std::vector<double>& u, const std::vector<double>& v)
  {
    check(wfx_wave_set_state(_wave, u.data(), v.data()));
  }
  // u_n, v_n after the solve (:282-285), host copies
  void solution(std::vector<double>& u_n, std::vector<double>& v_n) const
  {
    u_n.resize((std::size_t)_ndofs);
    v_n.resize((std::size_t)_ndofs);
    check(wfx_wave_get_state(_wave, u_n.data(), v_n.data()));
  }

  // perfectly matched layer (wavefx.h wfx_wave_set_pml, one rank): the layer of pml.zeta, built on the model's own
  // geometry from V (the space the model was made on); an empty zeta removes it.  psi and phi start at 0, as after
  // init and set_state.
  void set_pml(const SpaceView& V, const PML& pml)
  {
    if (!pml.zeta.empty() && (std::int64_t)pml.zeta.size() != 3 * _ndofs)
      throw std::runtime_error("wavefx: pml zeta needs 3 * ndofs entries");
    check(wfx_wave_set_pml(_wave, nullptr));
    wfx_pml_destroy(_pml);
    _pml = nullptr;
    _pml_cells = _pml_dofs = 0;
    if (pml.zeta.empty()) return;
    wfx_pml* h = nullptr;
    check(wfx_pml_create(_ctx->get(), _geom->get(), V.ndofs, V.dofmap, V.npoints, V.x, V.xdofs, pml.zeta.data(), &h));
    if (wfx_wave_set_pml(_wave, h))
    {
      wfx_pml_destroy(h);
      check(1);
    }
    _pml = h;
    check(wfx_pml_info(_pml, &_pml_cells, &_pml_dofs, nullptr));
  }
  // the layer's psi [layer dofs] and phi [layer cells][(P+1)^3][3] for checkpoints: get after solution(), set after
  // set_state()
  void pml_state(std::vector<double>& psi, std::vector<double>& phi) const
  {
    psi.resize((std::size_t)_pml_dofs);
    phi.resize((std::size_t)_pml_cells * _nq * 3);
    check(wfx_wave_get_pml_state(_wave, psi.data(), phi.data()));
  }
  void set_pml_state(const std::vector<double>& psi, const std::vector<double>& phi)
  {
    if ((std::int64_t)psi.size() != _pml_dofs || (std::int64_t)phi.size() != _pml_cells * _nq * 3)
      throw std::runtime_error("wavefx: pml state needs psi [layer dofs] and phi [layer cells][nq][3]");
    check(wfx_wave_set_pml_state(_wave, psi.data(), phi.data()));
  }

  std::shared_ptr<MassOperator<double>> mass_op;
  std::shared_ptr<StiffnessOperator<double>> stiff_op;
  // the C handle, e.g. for PennesGLL::heat_from_wave
  wfx_wave* get() const { return _wave; }
  std::int64_t ndofs() const { return _ndofs; }

protected:
  // the lossy / Westervelt models (wfx_wave_create_westervelt, one rank): see WesterveltGLLOpt
  LinearGLLOpt(std::shared_ptr<Context> ctx, const SpaceView& V, int degreeOfBasis, double speedOfSound,
               double sourceFrequency, double pressureAmplitude, double delta, double beta, double rho0,
               const Medium* medium = nullptr)
      : _ctx(std::move(ctx)), _ndofs(V.ndofs), _nq((std::int64_t)(V.degree + 1) * (V.degree + 1) * (V.degree + 1))
  {
    make_operators(V, degreeOfBasis, speedOfSound, medium);
    check(wfx_wave_create_westervelt(_ctx->get(), stiff_op->get(), mass_op->get(), _bnd, V.size_local, speedOfSound,
                                     sourceFrequency, pressureAmplitude, delta, beta, rho0, &_wave));
    if (medium && !medium->kappa.empty())
    {
      if ((std::int64_t)medium->kappa.size() != V.ndofs) throw std::runtime_error("wavefx: medium kappa needs ndofs entries");
      check(wfx_wave_set_nonlinearity(_wave, medium->kappa.data()));
    }
  }
  // geometry (scaled by the medium's stiffness weight), mass, stiffness and boundary operators of one rank
  void make_operators(const SpaceView& V, int degreeOfBasis, double speedOfSound, const Medium* medium)
  {
    _geom = std::make_shared<Geometry<double>>(_ctx, V);
    if (medium) check_medium(V, *medium);
    if (medium) _geom->scale_cells(medium->stiffness);
    mass_op = std::make_shared<MassOperator<double>>(_geom, V, degreeOfBasis, medium ? medium->mass.data() : nullptr);
    std::map<std::string, double> params{{"c0", speedOfSound}};
    stiff_op = std::make_shared<StiffnessOperator<double>>(_geom, V, degreeOfBasis, params);
    check(wfx_boundary_create_weighted(_ctx->get(), V.degree, WFX_F64, V.nfacets, V.facet_cell, V.facet_local,
                                       V.facet_tag, V.npoints, V.x, V.xdofs, V.ndofs, V.dofmap,
                                       medium ? medium->facet.data() : nullptr, &_bnd));
  }

private:
  static void snapshot_trampoline(void* self, std::int64_t step, double t, const void* u, const void* v)
  {
    auto* me = static_cast<LinearGLLOpt*>(self);
    if (me->_snap) me->_snap(step, t, static_cast<const double*>(u), static_cast<const double*>(v));
  }
  std::function<void(std::int64_t, double, const double*, const double*)> _snap;
  std::int64_t _nprobes = 0;
  std::shared_ptr<Context> _ctx;
  std::shared_ptr<VectorUpdater<double>> _halo;
  std::shared_ptr<Geometry<double>> _geom;
  std::int64_t _ndofs;
  wfx_boundary* _bnd = nullptr;
  wfx_wave* _wave = nullptr;
  wfx_pml* _pml = nullptr;
  std::int64_t _pml_cells = 0, _pml_dofs = 0, _nq = 0;
};
// The Westervelt model, one rank, fp64, with the interface of LinearGLLOpt (wavefx.h, DESIGN.md section 4.5a):
//   (1 - kappa p) p_tt - c0^2 lap p - delta lap p_t = kappa p_t^2,  kappa = 2 beta / (rho0 c0^2),
// dp/dn = g(t) on tag 1, dp/dn = -p_t / c0 on tag 2.  delta [m^2/s] >= 0, beta >= 0, rho0 > 0 when beta > 0.
class WesterveltGLLOpt : public LinearGLLOpt
{
public:
  WesterveltGLLOpt(std::shared_ptr<Context> ctx, const SpaceView& V, int degreeOfBasis, double speedOfSound,
                   double sourceFrequency, double pressureAmplitude, double diffusivityOfSound,
                   double coefficientOfNonlinearity, double density)
      : LinearGLLOpt(std::move(ctx), V, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                     diffusivityOfSound, coefficientOfNonlinearity, density)
  {
  }
  // in a layered medium: medium.kappa (per dof) in place of the scalar kappa when it is not empty
  WesterveltGLLOpt(std::shared_ptr<Context> ctx, const SpaceView& V, int degreeOfBasis, double speedOfSound,
                   double sourceFrequency, double pressureAmplitude, double diffusivityOfSound,
                   double coefficientOfNonlinearity, double density, const Medium& medium)
      : LinearGLLOpt(std::move(ctx), V, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                     diffusivityOfSound, coefficientOfNonlinearity, density, &medium)
  {
  }
  // a per-dof kappa (ndofs entries) in place of the scalar; an empty vector restores the scalar
  void set_nonlinearity(const std::vector<double>& kappa)
  {
    check(wfx_wave_set_nonlinearity(get(), kappa.empty() ? nullptr : kappa.data()));
  }
  // relaxation absorption (wavefx.h wfx_wave_set_relaxation, DESIGN.md section 4.5f): tau [M] > 0, eps [M][ndofs] >= 0
  // per dof (the Python Relaxation.eps_dofs); an empty tau switches it off.  The memory variables start at 0.
  void set_relaxation(const std::vector<double>& tau, const std::vector<double>& eps)
  {
    if (!tau.empty() && eps.size() != tau.size() * (std::size_t)ndofs())
      throw std::runtime_error("wavefx: relaxation eps needs M * ndofs entries");
    check(wfx_wave_set_relaxation(get(), (int)tau.size(), tau.empty() ? nullptr : tau.data(),
                                  tau.empty() ? nullptr : eps.data()));
    _relax_m = (int)tau.size();
  }
  // the memory variables q [M][ndofs], for checkpoints: get after solution(), set after set_state()
  void relaxation_state(std::vector<double>& q) const
  {
    q.resize((std::size_t)_relax_m * (std::size_t)ndofs());
    check(wfx_wave_get_relaxation_state(get(), q.data()));
  }
  void set_relaxation_state(const std::vector<double>& q)
  {
    if (q.size() != (std::size_t)_relax_m * (std::size_t)ndofs())
      throw std::runtime_error("wavefx: relaxation state needs M * ndofs entries");
    check(wfx_wave_set_relaxation_state(get(), q.data()));
  }

private:
  int _relax_m = 0;
};
// The lossy model: WesterveltGLLOpt with beta = 0,  p_tt - c0^2 lap p - delta lap p_t = 0
class LossyGLLOpt : public WesterveltGLLOpt
{
public:
  LossyGLLOpt(std::shared_ptr<Context> ctx, const SpaceView& V, int degreeOfBasis, double speedOfSound,
              double sourceFrequency, double pressureAmplitude, double diffusivityOfSound)
      : WesterveltGLLOpt(std::move(ctx), V, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                         diffusivityOfSound, 0.0, 1.0)
  {
  }
  LossyGLLOpt(std::shared_ptr<Context> ctx, const SpaceView& V, int degreeOfBasis, double speedOfSound,
              double sourceFrequency, double pressureAmplitude, double diffusivityOfSound, const Medium& medium)
      : WesterveltGLLOpt(std::move(ctx), V, degreeOfBasis, speedOfSound, sourceFrequency, pressureAmplitude,
                         diffusivityOfSound, 0.0, 1.0, medium)
  {
  }
};

// nv wave models on one mesh (1 <= nv <= WFX_ENSEMBLE_MAX), one rank, fp64: member m is
// LinearGLLOpt(V, degree, c0, f0[m], p0[m]); the stiffness apply of a stage reads G once for all members.
// States are member-interleaved [ndofs][nv] (entry (dof i, member m) at i*nv + m), probe values
// [nrec][nprobes][nv].  Snapshots are not available for ensembles.
class LinearGLLEnsemble
{
public:
  LinearGLLEnsemble(std::shared_ptr<Context> ctx, const SpaceView& V, int degreeOfBasis, double speedOfSound,
                    const std::vector<double>& sourceFrequencies, const std::vector<double>& pressureAmplitudes)
      : LinearGLLEnsemble(std::move(ctx), V, degreeOfBasis, speedOfSound, sourceFrequencies, pressureAmplitudes,
                          static_cast<const Medium*>(nullptr))
  {
  }
  // in a layered medium (its kappa is not used: the ensemble is linear)
  LinearGLLEnsemble(std::shared_ptr<Context> ctx, const SpaceView& V, int degreeOfBasis, double speedOfSound,
                    const std::vector<double>& sourceFrequencies, const std::vector<double>& pressureAmplitudes,
                    const Medium& medium)
      : LinearGLLEnsemble(std::move(ctx), V, degreeOfBasis, speedOfSound, sourceFrequencies, pressureAmplitudes,
                          &medium)
  {
  }

private:
  LinearGLLEnsemble(std::shared_ptr<Context> ctx, const SpaceView& V, int degreeOfBasis, double speedOfSound,
                    const std::vector<double>& sourceFrequencies, const std::vector<double>& pressureAmplitudes,
                    const Medium* medium)
      : _ctx(std::move(ctx)), _ndofs(V.ndofs), _nv((int)sourceFrequencies.size())
  {
    if (pressureAmplitudes.size() != sourceFrequencies.size())
      throw std::runtime_error("wavefx: one source frequency and one pressure amplitude per member expected");
    _geom = std::make_shared<Geometry<double>>(_ctx, V);
    if (medium) check_medium(V, *medium);
    if (medium) _geom->scale_cells(medium->stiffness);
    mass_op = std::make_shared<MassOperator<double>>(_geom, V, degreeOfBasis, medium ? medium->mass.data() : nullptr);
    std::map<std::string, double> params{{"c0", speedOfSound}};
    stiff_op = std::make_shared<StiffnessOperator<double>>(_geom, V, degreeOfBasis, params, std::vector<std::int32_t>{},
                                                           WFX_STIFF_ENSEMBLE);
    check(wfx_boundary_create_weighted(_ctx->get(), V.degree, WFX_F64, V.nfacets, V.facet_cell, V.facet_local,
                                       V.facet_tag, V.npoints, V.x, V.xdofs, V.ndofs, V.dofmap,
                                       medium ? medium->facet.data() : nullptr, &_bnd));
    check(wfx_wave_create_ensemble(_ctx->get(), stiff_op->get(), mass_op->get(), _bnd, _nv, V.size_local, speedOfSound,
                                   sourceFrequencies.data(), pressureAmplitudes.data(), &_wave));
  }

public:
  ~LinearGLLEnsemble()
  {
    wfx_wave_destroy(_wave);
    wfx_boundary_destroy(_bnd);
  }
  LinearGLLEnsemble(const LinearGLLEnsemble&) = delete;
  LinearGLLEnsemble& operator=(const LinearGLLEnsemble&) = delete;

  int size() const { return _nv; }
  void init() { check(wfx_wave_init(_wave)); }
  // device arrays of ndofs * nv entries
  void f0(double t, const double* u_dev, const double* v_dev, double* result_dev, void* stream = nullptr)
  {
    check(wfx_wave_f0(_wave, t, u_dev, v_dev, result_dev, stream));
  }
  void f1(double t, const double* u_dev, const double* v_dev, double* result_dev, void* stream = nullptr)
  {
    check(wfx_wave_f1(_wave, t, u_dev, v_dev, result_dev, stream));
  }
  std::int64_t rk4(double startTime, double finalTime, double timeStep)
  {
    std::int64_t steps = 0;
    double t_end = 0;
    check(wfx_wave_rk4(_wave, startTime, finalTime, timeStep, 0, &steps, &t_end, nullptr));
    _ctx->synchronize();
    return steps;
  }
  void set_probes(const std::vector<std::int32_t>& dofs, std::int64_t max_records)
  {
    _nprobes = (std::int64_t)dofs.size();
    check(wfx_wave_set_probes(_wave, _nprobes, dofs.data(), max_records));
  }
  // times [nrec] and values [nrec][nprobes][nv] recorded so far
  void probe_series(std::vector<double>& t, std::vector<double>& values) const
  {
    std::int64_t n = 0;
    check(wfx_wave_get_probe_series(_wave, &n, nullptr, nullptr));
    t.resize((std::size_t)n);
    values.resize((std::size_t)(n * _nprobes * _nv));
    check(wfx_wave_get_probe_series(_wave, &n, t.data(), values.data()));
  }
  // as LinearGLLOpt's, member m analysed at its own f0[m]; peaks [ndofs][nv], harmonics [nharm][ndofs][nv]
  void set_field_stats(bool enable, double t_start = 0.0, int nharm = 0)
  {
    check(wfx_wave_set_field_stats(_wave, enable ? 1 : 0, t_start, nharm));
  }
  void field_stats(FieldStats& out) const { read_field_stats(_wave, _ndofs * _nv, out); }
  // as LinearGLLOpt's, member m with its own profile: amp, delay [ndofs][nv] (member-interleaved)
  void set_source_profile(const std::vector<double>& amp, const std::vector<double>& delay)
  {
    set_profile(_wave, _ndofs * _nv, amp, delay);
  }
  // as LinearGLLOpt's, a column per member: q, delay [dofs][nv] (member-interleaved)
  void set_volume_source(const std::vector<std::int32_t>& dofs, const std::vector<double>& q,
                         const std::vector<double>& delay)
  {
    set_volume(_wave, _nv, dofs, q, delay);
  }
  void set_state(const std::vector<double>& u, const std::vector<double>& v)
  {
    if ((std::int64_t)u.size() != _ndofs * _nv || (std::int64_t)v.size() != _ndofs * _nv)
      throw std::runtime_error("wavefx: ensemble state must hold ndofs * nv entries");
    check(wfx_wave_set_state(_wave, u.data(), v.data()));
  }
  void solution(std::vector<double>& u_n, std::vector<double>& v_n) const
  {
    u_n.resize((std::size_t)(_ndofs * _nv));
    v_n.resize((std::size_t)(_ndofs * _nv));
    check(wfx_wave_get_state(_wave, u_n.data(), v_n.data()));
  }

  std::shared_ptr<MassOperator<double>> mass_op;
  std::shared_ptr<StiffnessOperator<double>> stiff_op;

private:
  std::shared_ptr<Context> _ctx;
  std::shared_ptr<Geometry<double>> _geom;
  std::int64_t _ndofs;
  int _nv;
  std::int64_t _nprobes = 0;
  wfx_boundary* _bnd = nullptr;
  wfx_wave* _wave = nullptr;
};

// The Pennes bioheat model with a CEM43 thermal dose (wfx_thermal_create, DESIGN.md section 4.5d), one rank, fp64:
//   rhoC T_t = div(k grad T) - wbCb (T - T_art) + s Q,   -k dT/dn = h[j] (T - T_ext[j]) on tag j + 1
// rhoC and wbCb per dof (mass-weighted averages of per-cell values, INTEGRATION.md; an empty perfusion is 0).
// Temperatures in and out are absolute (T = T_art + theta).  T_ext: the two Robin tags' exterior temperatures, nullptr
// for T_art on both.
class PennesGLL
{
public:
  PennesGLL(std::shared_ptr<Context> ctx, const SpaceView& V, int degree, double k, const std::vector<double>& rhoC,
            const std::vector<double>& perfusion, double T_art, std::array<double, 2> h = {0.0, 0.0},
            const std::array<double, 2>* T_ext = nullptr)
      : _ctx(std::move(ctx)), _ndofs(V.ndofs), _T_art(T_art)
  {
    if ((std::int64_t)rhoC.size() != _ndofs || (!perfusion.empty() && (std::int64_t)perfusion.size() != _ndofs))
      throw std::runtime_error("wavefx: rhoC and perfusion must hold one value per dof");
    _geom = std::make_shared<Geometry<double>>(_ctx, V);
    mass_op = std::make_shared<MassOperator<double>>(_geom, V, degree);
    std::map<std::string, double> params; // the stiffness operator's own c0 (1500) is folded into the scale
    stiff_op = std::make_shared<StiffnessOperator<double>>(_geom, V, degree, params);
    if (h[0] != 0.0 || h[1] != 0.0)
      check(wfx_boundary_create(_ctx->get(), V.degree, WFX_F64, V.nfacets, V.facet_cell, V.facet_local, V.facet_tag,
                                V.npoints, V.x, V.xdofs, V.ndofs, V.dofmap, &_bnd));
    check(wfx_thermal_create(_ctx->get(), stiff_op->get(), mass_op->get(), _bnd, k, rhoC.data(),
                             perfusion.empty() ? nullptr : perfusion.data(), T_art, h.data(), T_ext ? T_ext->data() : nullptr, &_th));
  }
  ~PennesGLL()
  {
    wfx_thermal_destroy(_th);
    wfx_boundary_destroy(_bnd);
  }
  PennesGLL(const PennesGLL&) = delete;
  PennesGLL& operator=(const PennesGLL&) = delete;

  void init() { check(wfx_thermal_init(_th)); }
  void set_temperature(const std::vector<double>& T)
  {
    if ((std::int64_t)T.size() != _ndofs) throw std::runtime_error("wavefx: one temperature per dof expected");
    std::vector<double> rise(T.size());
    for (std::size_t i = 0; i < T.size(); ++i) rise[i] = T[i] - _T_art;
    check(wfx_thermal_set_state(_th, rise.data()));
  }
  void temperature(std::vector<double>& T) const
  {
    T.resize((std::size_t)_ndofs);
    check(wfx_thermal_get_state(_th, T.data()));
    for (double& x : T) x += _T_art;
  }
  // Q [W/m^3] per dof; empty: 0
  void set_heat_source(const std::vector<double>& Q) { check(wfx_thermal_set_heat_source(_th, Q.empty() ? nullptr : Q.data())); }
  void heat_source(std::vector<double>& Q) const
  {
    Q.resize((std::size_t)_ndofs);
    check(wfx_thermal_get_heat_source(_th, Q.data()));
  }
  // Q from the harmonic maps of a wave model's field statistics, alpha(f) = alpha0 (f / 1 MHz)^y
  void heat_from_wave(const LinearGLLOpt& wave, double alpha0, double y, double rho0, double c0)
  {
    check(wfx_thermal_heat_from_wave(_th, wave.get(), 0, alpha0, nullptr, y, rho0, c0));
  }
  void set_heat_scale(double s) { check(wfx_thermal_set_heat_scale(_th, s)); }
  std::int64_t rk4(double startTime, double finalTime, double timeStep)
  {
    std::int64_t steps = 0;
    double t_end = 0;
    check(wfx_thermal_rk4(_th, startTime, finalTime, timeStep, 0, &steps, &t_end, nullptr));
    _ctx->synchronize();
    return steps;
  }
  // steps since init / set_temperature, CEM43 [min] and the peak temperature of every dof
  std::int64_t dose(std::vector<double>& cem43, std::vector<double>& T_max) const
  {
    std::int64_t n = 0;
    cem43.resize((std::size_t)_ndofs);
    T_max.resize((std::size_t)_ndofs);
    check(wfx_thermal_get_dose(_th, &n, cem43.data(), T_max.data()));
    for (double& x : T_max) x += _T_art;
    return n;
  }
  // safety * the power iteration's RK4 limit; the estimate approaches the limit from above, hence the safety factor
  double stable_dt(double safety = 0.8, int iters = 200) const
  {
    double lambda = 0, dt_max = 0;
    check(wfx_thermal_stable_dt(_th, iters, &lambda, &dt_max));
    return safety * dt_max;
  }

  std::shared_ptr<MassOperator<double>> mass_op;
  std::shared_ptr<StiffnessOperator<double>> stiff_op;

private:
  std::shared_ptr<Context> _ctx;
  std::shared_ptr<Geometry<double>> _geom;
  std::int64_t _ndofs;
  double _T_art;
  wfx_boundary* _bnd = nullptr;
  wfx_thermal* _th = nullptr;
};
} // namespace wavefx
