// Internal declarations shared by the libwavefx translation units.
#pragma once

#include "wavefx.h"

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#define WFX_MAXN 12 // max GLL points per direction handled by the host tables

struct wfx_stiffness;
struct wfx_halo;

namespace wfx
{
void set_error(const char* fmt, ...);

struct Error : std::runtime_error
{
  using std::runtime_error::runtime_error;
};

[[noreturn]] void fail(const char* fmt, ...);

#define WFX_CUDA(call)                                                                           \
  do                                                                                             \
  {                                                                                              \
    cudaError_t e_ = (call);                                                                     \
    if (e_ != cudaSuccess)                                                                       \
      wfx::fail("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));      \
  } while (0)

// Body wrapper for every extern "C" entry point: exceptions -> status + message.
#define WFX_API_BEGIN try {
#define WFX_API_END                                                                              \
  return 0;                                                                                      \
  }                                                                                              \
  catch (const std::exception& e)                                                                \
  {                                                                                              \
    wfx::set_error("%s", e.what());                                                              \
    return 1;                                                                                    \
  }                                                                                              \
  catch (...)                                                                                    \
  {                                                                                              \
    wfx::set_error("unknown error");                                                             \
    return 2;                                                                                    \
  }

// RAII device buffer (role of cuda::array<T>, common/cuda/array.hpp, without its
// implicit-copy double free).
template <typename T>
struct DevBuf
{
  T* p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  explicit DevBuf(size_t n_) { alloc(n_); }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept
  {
    if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
    return *this;
  }
  ~DevBuf() { release(); }
  void alloc(size_t n_)
  {
    release();
    // n is set once the allocation succeeded: after a failed one the buffer is empty, not sized with p = NULL
    if (n_) WFX_CUDA(cudaMalloc((void**)&p, n_ * sizeof(T)));
    n = n_;
  }
  void release()
  {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  void upload(const T* h, size_t cnt)
  {
    if (cnt > n) alloc(cnt);
    if (cnt) WFX_CUDA(cudaMemcpy(p, h, cnt * sizeof(T), cudaMemcpyHostToDevice));
  }
  void upload(const std::vector<T>& h) { upload(h.data(), h.size()); }
  void download(T* h, size_t cnt) const
  {
    if (cnt) WFX_CUDA(cudaMemcpy(h, p, cnt * sizeof(T), cudaMemcpyDeviceToHost));
  }
};

// host tables (wfx_tables.cpp)
void gll_points_weights(int P, double* pts, double* wts); // [0,1,interior] ordering
void deriv_1d(int P, double* D, bool clamp);              // D[q*n+i]
void tensor_perm(int P, int32_t* perm);                   // tensor index -> DOLFINx dof
double clamp_m101(double v);                              // xt::isclose clamp to -1/0/1

int stiffness_dtype(const struct ::wfx_stiffness* op);    // wfx_stiffness.cu
bool stiffness_has_split(const struct ::wfx_stiffness* op); // interface/interior parts present
bool stiffness_graph_safe(const struct ::wfx_stiffness* op); // its launches may be captured into a CUDA graph
int halo_dtype(const struct ::wfx_halo* h);                // wfx_halo.cu
bool mass_assembled(const struct ::wfx_mass* op);          // wfx_mass.cu: diagonal summed over the ranks
int mass_dtype(const struct ::wfx_mass* op);
int64_t mass_ndofs(const struct ::wfx_mass* op);          // length of the diagonal
bool boundary_assembled(const struct ::wfx_boundary* op);  // wfx_boundary.cu: facet masses summed over the ranks
int boundary_dtype(const struct ::wfx_boundary* op);
int64_t boundary_ndofs(const struct ::wfx_boundary* op);  // length of the vectors it adds into
// wfx_boundary_apply with the source amplitude g read from device memory at run time (CUDA-graph
// replays of a time step change g without touching the graph), wfx_boundary.cu
void boundary_apply_dev(struct ::wfx_boundary* op, double c0, const double* g_dev, const void* vn, void* b,
                        cudaStream_t stream);
// ensemble models (member-interleaved vectors [ndofs][nv]): the operator has the ensemble path
// (wfx_stiffness.cu); boundary term of every member, b[i,m] += c0^2 g_m m1_i - c0 m2_i vn[i,m], with the nv
// amplitudes from g_dev when it is not NULL (graph replays), else from g_host (wfx_boundary.cu)
bool stiffness_has_ensemble(const struct ::wfx_stiffness* op);
void boundary_apply_ens(struct ::wfx_boundary* op, int nv, double c0, const double* g_host, const double* g_dev,
                        const void* vn, void* b, cudaStream_t stream);
// source profiles (wfx_wave_set_source_profile, DESIGN.md section 4.5c): the compact dof list of the boundary
// term (the order of its amp / delay arrays), and the term with per-entry delayed sources
//   b[i,m] += c0^2 amp[t] (g_m + s_src g_m')(tn - delay[t]) m1_i - c0 m2_i vn[i,m],  t = p nv + m, i = dofs[p],
// g_m from member m's f0 / p0 (nv = 1: one field); tn read from t_dev when it is not NULL (graph replays)
struct SourceParams
{
  double f0[WFX_ENSEMBLE_MAX], p0[WFX_ENSEMBLE_MAX];
};
const std::vector<int32_t>& boundary_dofs(const struct ::wfx_boundary* op);
void boundary_apply_profile(struct ::wfx_boundary* op, int nv, double c0, double s_src, const SourceParams& sp,
                            double t_host, const double* t_dev, const double* amp, const double* delay,
                            const void* vn, void* b, cudaStream_t stream);
// volume sources (wfx_wave_set_volume_source, DESIGN.md section 4.5h): ns distinct dofs idx [ns] (device), weights q and
// delays [ns][nv] (device, fp64),
//   b[idx[p],m] += c0^2 q[t] g_m(tn - delay[t]),  t = p nv + m,  g_m = 0 before the delay,
// g_m from member m's f0 / p0 (nv = 1: one field); tn read from t_dev when it is not NULL (graph replays)
void volume_source_apply(int dtype, int64_t ns, int nv, const int32_t* idx, const double* q, const double* delay,
                         double c0, const SourceParams& sp, double t_host, const double* t_dev, void* b,
                         cudaStream_t stream);
// lossy / Westervelt models (wfx_wave_create_westervelt)
double stiffness_c0(const struct ::wfx_stiffness* op);       // the c0 of y = -c0^2 K x
int64_t stiffness_nshared(const struct ::wfx_stiffness* op); // rank-shared dofs (0 on one rank)
const double* mass_diagonal64(const struct ::wfx_mass* op);   // m on the device, fp64 whatever the dtype
// On the absorbing (tag 2) dofs: b_i -> m_i [kv_i (1 - kappa p_i) - kappa pd_i^2] with the exact
// kv_i = (b_i + kappa m_i pd_i^2) / (m_i (1 - kappa p_i) + qc m2_i), so that the dense stage update
// kv = (b minv + kappa pd^2) / (1 - kappa p) yields it; p = pw - s pd (s = 0: pw is p itself).  kappa_b (nullable):
// a per-dof kappa in fp64, compact over boundary_dofs(op), in place of the scalar kappa
void boundary_absorbing_mass(struct ::wfx_boundary* op, const double* m64, double qc, double kappa,
                             const double* kappa_b, double s, const void* pw, const void* pd, void* b,
                             cudaStream_t stream);
// Relaxation processes (wfx_wave_set_relaxation, DESIGN.md section 4.5f): 1 / tau_nu of the M processes
struct RelaxTau
{
  double inv_tau[WFX_RELAX_MAX];
};
// boundary_absorbing_mass with M relaxation processes: b_i -> m_i [kv_i (1 - kappa p_i) - kappa pd_i^2 + R_i] with
// the exact kv_i = (b_i + m_i (kappa pd_i^2 - R_i)) / (m_i (1 - kappa p_i) + qc m2_i), R_i = sum_nu q_nu,i'' from the
// stage's memory variables q [M][ndofs] (model dtype) and eps_b [M][nb] (fp64, compact over boundary_dofs(op))
void boundary_absorbing_mass_relax(struct ::wfx_boundary* op, const double* m64, double qc, double kappa,
                                   const double* kappa_b, int M, const RelaxTau& rt, const double* eps_b, const void* q,
                                   double s, const void* pw, const void* pd, void* b, cudaStream_t stream);
// A wave model's field statistics as the thermal model reads them (wfx_thermal_heat_from_wave, DESIGN.md section
// 4.5d): the unscaled fp64 harmonic sums, planes [h][ndofs * nv] (entry (dof i, member m) at i nv + m), the number
// of sampled steps N (the amplitudes are the sums times 2 / N) and every member's source frequency (wfx_wave.cu)
struct WaveFieldStats
{
  wfx_ctx* ctx = nullptr;
  int64_t ndofs = 0;
  int nv = 1;
  bool on = false;
  int nharm = 0;
  int64_t nsamples = 0;
  const double2* harm = nullptr;
  double f0[WFX_ENSEMBLE_MAX] = {};
};
WaveFieldStats wave_field_stats(const struct ::wfx_wave* w);

// Perfectly matched layer (wfx_pml_create, DESIGN.md section 4.5g), wfx_pml.cu.  One RK4 stage (update = true) or the
// right-hand side of f1 (update = false, stage 0): adds the layer's terms to b and steps psi and phi.  Vectors in the
// model dtype: w the stiffness input, p = u_ at stage 0 (v_ its rate) and w - s vn at stages 1-3; psi [npd] and phi
// [cells][3][nq] (solution _, start of step 0, stage state n), r [cells][nq] scratch, m the mass m~ compact [npd].
struct PmlStage
{
  int stage = 0;
  bool update = true;
  double cK2 = 0, s = 0, bdt = 0, adt = 0;
  const void *w = nullptr, *u_ = nullptr, *v_ = nullptr, *vn = nullptr, *m = nullptr;
  void *psi_ = nullptr, *psi0 = nullptr, *psin = nullptr, *phi_ = nullptr, *phi0 = nullptr, *phin = nullptr;
  void *r = nullptr, *b = nullptr;
};
void pml_stage(const struct ::wfx_pml* pm, const PmlStage& q, cudaStream_t st);
// wfx_geometry_scale_cells on a registered layer: its per-cell coefficients times coeff_host[geometry cell]
void pml_scale_cells(struct ::wfx_pml* pm, const double* coeff_host);
// what a wave model needs to know of a layer to take it (wfx_wave_set_pml)
struct PmlShape
{
  wfx_ctx* ctx = nullptr;
  const struct ::wfx_geom* geom = nullptr;
  int dtype = 0, nq = 0;
  int64_t ndofs = 0, ncells = 0, npd = 0;
  double zeta_max = 0;
  const std::vector<int32_t>* dofs = nullptr; // global dof of each PML dof
};
PmlShape pml_shape(const struct ::wfx_pml* pm);
const struct ::wfx_geom* stiffness_geom(const struct ::wfx_stiffness* op); // wfx_stiffness.cu

// NVTX ranges around the phases of a time step (the reference marks its profiled regions the same
// way: demo/gpu_scatter_mpi/main.cpp:101-121, demo/gpu_cg/CUDA/cg.hpp:74-113).  nvtx3 is header-only
// and costs a few nanoseconds when no tool is attached.
struct NvtxRange
{
  explicit NvtxRange(const char* name);
  ~NvtxRange();
};

// Set-up phase timer: WFX_VERBOSE=1 prints the seconds spent per phase of the create calls to stderr.
struct SetupTimer
{
  explicit SetupTimer(const char* what);
  void lap(const char* phase);
  const char* what;
  double last;
  bool on;
};

struct ScopedDevice
{
  int prev = -1;
  explicit ScopedDevice(int dev)
  {
    cudaGetDevice(&prev);
    if (prev != dev) WFX_CUDA(cudaSetDevice(dev));
  }
  ~ScopedDevice() { if (prev >= 0) cudaSetDevice(prev); }
};
} // namespace wfx

struct wfx_ctx
{
  int device = 0;
  int num_sms = 0;
  size_t smem_optin = 0;
};

// Geometric factors on the device (kernel layout).
//   nq = n^3 points per cell, n = P+1, n2 = n^2.
//   point index inside a cell is "k-major": r = k*n2 + (i*n + j) for tensor node (i,j,k)
//   (i <-> x, slowest in the reference's tensor order; k <-> z).
//   G6  [ncells][n][3][n2][2]  per k-plane three pairs (00,01) (02,11) (12,22) per column, dtype T;
//       column of point (i,j) is i*n+j unless g_colpos is set (a stiffness operator may reorder
//       the columns once, in place, to the lane order of its kernel: wfx_stiffness.cu)
//   dJw [ncells][nq]     detJ * w, fp64 (setup-only consumers)
struct wfx_geom
{
  wfx_ctx* ctx = nullptr;
  int P = 0, n = 0, nq = 0, dtype = WFX_F64;
  int64_t ncells = 0;
  void* G6 = nullptr;     // T
  std::vector<uint8_t> g_colpos; // empty: identity; else column of point (i,j) = g_colpos[i*n+j]
  // private copies of G6 that stiffness operators made from it ([ncells][nq*6] T each, cell-major; the
  // points inside a cell may be reordered): wfx_geometry_scale_cells scales them with G6, so a coefficient
  // set after an operator was created reaches every path.  An operator registers its copy at creation and
  // removes it when destroyed.
  std::vector<void*> g_copies;
  // the composed wfx_geometry_scale_cells coefficient per cell (empty: never scaled), and the perfectly matched
  // layers built on this geometry, which it scales the same way (a layer reads it at creation and registers itself)
  std::vector<double> cell_coeff;
  std::vector<struct ::wfx_pml*> pmls;
  double* dJw = nullptr;  // fp64
  // Affine cells (parallelepipeds): G[c,q] = w_q * A_c with one symmetric 3x3 A_c per cell.  Detected
  // from the computed (clamped) per-point G, so a cell counts as affine only if the per-cell form
  // reproduces the reference's values to rounding.  Gc [ncells][6] (00,01,02,11,12,22), dtype T,
  // meaningful where affine[c] != 0; n_affine == ncells selects the stiffness kernels that never
  // read G6 (structured fast path).
  void* Gc = nullptr;
  uint8_t* affine = nullptr;  // device [ncells]
  int64_t n_affine = 0;
  // cell centroids (host) for the locality-preserving batch plan
  std::vector<float> centroid; // [ncells][3]
  // exact integer grid coordinates from the connectivity when the mesh is one structured block
  // (wfx_plan.h structured_cell_coords), else empty
  std::vector<int32_t> cell_ijk; // [ncells][3]
  ~wfx_geom();
};
