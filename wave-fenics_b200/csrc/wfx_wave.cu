// Wave model and classical RK4 time integrator on the device.
// Replaces LinearGLLOpt::{init,f0,f1,rk4} (common/LinearGLL.hpp:131-287).  The reference
// makes ~17 full-vector passes per stage (copies, axpys, zero, divide) plus three host
// MPI scatters; here a stage is: stiffness apply (b = -c0^2 K un), boundary term on the
// facet dofs, one optional halo reduction of b, and ONE fused pointwise kernel that does
// kv = b/m, both solution updates and the next stage state.
#include "wfx_internal.h"
#include "wfx_source.h"

#include <cmath>
#include <cstdlib>

using namespace wfx;

struct wfx_stiffness;
struct wfx_mass;
struct wfx_boundary;
struct wfx_halo;

struct wfx_wave
{
  wfx_ctx* ctx = nullptr;
  wfx_stiffness* stiff = nullptr;
  wfx_mass* mass = nullptr;
  wfx_boundary* bnd = nullptr;
  wfx_halo* halo = nullptr;
  int dtype = WFX_F64;
  int64_t n = 0, size_local = 0;
  double c0 = 0, f0 = 0, p0 = 0;
  // ensemble model (wfx_wave_create_ensemble): nv members, vectors [n][nv], member m's source (f0s[m], p0s[m])
  bool ens = false;
  int nv = 1;
  std::vector<double> f0s, p0s;
  // lossy (model 1) and Westervelt (model 2) models (wfx_wave_create_westervelt).  The stiffness input
  // w = u + s_stiff v lives in `un` (nothing else reads un in these models); the source passed to the
  // boundary term is g + s_src g'; q = qc m2 is the Gamma2 mass term; f1 builds its w in f1_w.
  int model = 0;
  double kappa = 0, s_stiff = 0, s_src = 0, qc = 0;
  const double* m64 = nullptr;
  DevBuf<unsigned char> f1_w;
  const void* minv = nullptr;
  // u_, v_: solution; u0, v0: start of step; un, vn: stage state; b: right-hand side
  DevBuf<unsigned char> u_, v_, u0, v0, un, vn, b;
  // distributed runs: the ghost reduction runs on its own stream, ordered by events
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t ev_iface = nullptr, ev_halo = nullptr;
  // one-rank runs: a full time step (4 stages, ~40 launches) is captured once per step size
  // into a CUDA graph and replayed; the four source amplitudes of the step live in g_dev
  // ([stage][member] for an ensemble)
  bool use_graph = true;
  cudaGraphExec_t step_graph = nullptr;
  double graph_dt = 0;
  DevBuf<double> g_dev;
  // source profile (section 4.5c): per-entry amplitude and delay, compact over the boundary dofs [nb][nv]; the
  // boundary term then evaluates the delayed sources on the device from the four stage times, which graph
  // replays read from t_dev.  Setting or clearing it drops step_graph (captured with the other boundary kernel).
  bool prof_on = false;
  DevBuf<double> prof_amp, prof_delay, t_dev;
  cudaStream_t own_stream = nullptr; // capture needs a non-legacy stream
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  // time-stepping position (reset by init / set_state): steps completed and the time reached
  int64_t steps_done = 0;
  double t_now = 0;
  // probes: u at selected dofs after every completed step, kept on the device until asked for
  int64_t nprobes = 0, probe_cap = 0, probe_rec = 0;
  DevBuf<int32_t> d_probe_idx;
  DevBuf<unsigned char> d_probe_val;
  std::vector<double> probe_t;
  // field statistics (section 4.5b): peaks [n*nv] in the model dtype and stats_nharm double2 planes [h][n*nv] of
  // fp64 harmonic sums, updated after every step with t_n >= stats_t_start - dt/2; reset with the probes
  bool stats_on = false;
  int stats_nharm = 0;
  double stats_t_start = 0, stats_t_first = 0, stats_t_last = 0;
  int64_t stats_n = 0;
  DevBuf<unsigned char> stats_pmax, stats_pmin;
  DevBuf<double2> stats_harm;
  // snapshots: every `snap_every` steps u, v are copied device -> device on the work stream, then
  // device -> pinned host on a copy stream while the time stepping goes on; the callback runs on the
  // calling thread once the copy has landed (at the next snapshot or at the end of rk4)
  int64_t snap_every = 0;
  wfx_snapshot_fn snap_fn = nullptr;
  void* snap_user = nullptr;
  DevBuf<unsigned char> snap_u, snap_v;
  void *snap_hu = nullptr, *snap_hv = nullptr; // pinned
  cudaStream_t snap_stream = nullptr;
  cudaEvent_t ev_snap_ready = nullptr, ev_snap_done = nullptr;
  bool snap_pending = false;
  int64_t snap_step = 0;
  double snap_t = 0;
  ~wfx_wave()
  {
    if (snap_hu) cudaFreeHost(snap_hu);
    if (snap_hv) cudaFreeHost(snap_hv);
    if (snap_stream) cudaStreamDestroy(snap_stream);
    if (ev_snap_ready) cudaEventDestroy(ev_snap_ready);
    if (ev_snap_done) cudaEventDestroy(ev_snap_done);
    if (step_graph) cudaGraphExecDestroy(step_graph);
    if (own_stream) cudaStreamDestroy(own_stream);
    if (ev_in) cudaEventDestroy(ev_in);
    if (ev_out) cudaEventDestroy(ev_out);
    if (ev_iface) cudaEventDestroy(ev_iface);
    if (ev_halo) cudaEventDestroy(ev_halo);
    if (comm_stream) cudaStreamDestroy(comm_stream);
  }
};

namespace
{
// Stage update, fused (SURVEY.md App. C.3).  STAGE 0 reads the solution as stage state
// and saves it as u0/v0; STAGE 3 only finishes the solution.
//   kv = b / m                          (LinearGLL.hpp:188-191; m^-1 precomputed, :179-181)
//   u_ += b_i dt ku,  v_ += b_i dt kv   (:264-265), ku = vn (f0, :141-144)
//   un' = u0 + a_{i+1} dt ku, vn' = v0 + a_{i+1} dt kv   (:250-254 of the next stage)
template <typename T, int STAGE>
__global__ void __launch_bounds__(256)
rk_stage_kernel(int64_t n, const T* __restrict__ b, const T* __restrict__ minv, T* __restrict__ u_,
                T* __restrict__ v_, T* __restrict__ u0, T* __restrict__ v0, T* __restrict__ un,
                T* __restrict__ vn, T bdt, T adt_next)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n) return;
  const T kv = b[k] * minv[k];
  T us = u_[k], vs = v_[k];
  T ku, ub, vb;
  if (STAGE == 0)
  {
    ku = vs;
    ub = us;
    vb = vs;
    u0[k] = ub;
    v0[k] = vb;
  }
  else
  {
    ku = vn[k];
    if (STAGE < 3)
    {
      ub = u0[k];
      vb = v0[k];
    }
  }
  u_[k] = ku * bdt + us;
  v_[k] = kv * bdt + vs;
  if (STAGE < 3)
  {
    un[k] = ku * adt_next + ub;
    vn[k] = kv * adt_next + vb;
  }
}

template <typename T>
void launch_stage(int stage, int64_t n, const void* b, const void* minv, void* u_, void* v_,
                  void* u0, void* v0, void* un, void* vn, double bdt, double adt_next,
                  cudaStream_t st)
{
  const unsigned grid = (unsigned)((n + 255) / 256);
#define WFX_STAGE(S)                                                                             \
  rk_stage_kernel<T, S><<<grid, 256, 0, st>>>(n, (const T*)b, (const T*)minv, (T*)u_, (T*)v_,   \
                                               (T*)u0, (T*)v0, (T*)un, (T*)vn, (T)bdt, (T)adt_next)
  switch (stage)
  {
  case 0: WFX_STAGE(0); break;
  case 1: WFX_STAGE(1); break;
  case 2: WFX_STAGE(2); break;
  default: WFX_STAGE(3); break;
  }
#undef WFX_STAGE
  WFX_CUDA(cudaGetLastError());
}
// rk_stage_kernel on member-interleaved vectors, one thread per entry: the nv threads of a dof are adjacent
// lanes, so every access of a warp is contiguous and minv[i] is one broadcast load for all members of dof i
template <typename T, int STAGE>
__global__ void __launch_bounds__(256)
rk_stage_ens_kernel(int64_t n, int nv, const T* __restrict__ b, const T* __restrict__ minv, T* __restrict__ u_,
                    T* __restrict__ v_, T* __restrict__ u0, T* __restrict__ v0, T* __restrict__ un,
                    T* __restrict__ vn, T bdt, T adt_next)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n * nv) return;
  const T kv = b[k] * minv[k / nv];
  T us = u_[k], vs = v_[k];
  T ku, ub, vb;
  if (STAGE == 0)
  {
    ku = vs;
    ub = us;
    vb = vs;
    u0[k] = ub;
    v0[k] = vb;
  }
  else
  {
    ku = vn[k];
    if (STAGE < 3)
    {
      ub = u0[k];
      vb = v0[k];
    }
  }
  u_[k] = ku * bdt + us;
  v_[k] = kv * bdt + vs;
  if (STAGE < 3)
  {
    un[k] = ku * adt_next + ub;
    vn[k] = kv * adt_next + vb;
  }
}

template <typename T>
void launch_stage_ens(int stage, int64_t n, int nv, const void* b, const void* minv, void* u_, void* v_, void* u0,
                      void* v0, void* un, void* vn, double bdt, double adt_next, cudaStream_t st)
{
  const unsigned grid = (unsigned)((n * nv + 255) / 256);
#define WFX_STAGE(S)                                                                                        \
  rk_stage_ens_kernel<T, S><<<grid, 256, 0, st>>>(n, nv, (const T*)b, (const T*)minv, (T*)u_, (T*)v_,     \
                                                   (T*)u0, (T*)v0, (T*)un, (T*)vn, (T)bdt, (T)adt_next)
  switch (stage)
  {
  case 0: WFX_STAGE(0); break;
  case 1: WFX_STAGE(1); break;
  case 2: WFX_STAGE(2); break;
  default: WFX_STAGE(3); break;
  }
#undef WFX_STAGE
  WFX_CUDA(cudaGetLastError());
}

// Stage update of the lossy (NL = false) and Westervelt (NL = true) models: rk_stage_kernel, and
//   kv = b / m                                          (lossy)
//   kv = (b / m + kappa pd^2) / (1 - kappa p)           (Westervelt; pd = ku = the stage's v)
//   w' = un' + s vn'  written where rk_stage_kernel writes un'; STAGE 3 writes w = u_ + s v_ for the next step.
// p is u_ at stage 0; at stages 1-3 it is rebuilt as w - s vn (one read of w, no un vector).
// On the absorbing dofs b has been replaced beforehand (boundary_absorbing_mass) so that this
// quotient is the exact kv of the lumped system with the Gamma2 mass term.
template <typename T, int STAGE, bool NL>
__global__ void __launch_bounds__(256)
rk_stage_westervelt_kernel(int64_t n, const T* __restrict__ b, const T* __restrict__ minv, T* __restrict__ u_,
                           T* __restrict__ v_, T* __restrict__ u0, T* __restrict__ v0, T* __restrict__ w,
                           T* __restrict__ vn, T bdt, T adt_next, T s, T kappa)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n) return;
  T kv = b[k] * minv[k];
  T us = u_[k], vs = v_[k];
  T ku, ub, vb, p;
  if (STAGE == 0)
  {
    ku = vs;
    ub = us;
    vb = vs;
    p = us;
    u0[k] = ub;
    v0[k] = vb;
  }
  else
  {
    ku = vn[k];
    if (NL) p = w[k] - s * ku;
    if (STAGE < 3)
    {
      ub = u0[k];
      vb = v0[k];
    }
  }
  if (NL) kv = (kv + kappa * ku * ku) / (T(1) - kappa * p);
  const T un_ = ku * bdt + us, vn_ = kv * bdt + vs;
  u_[k] = un_;
  v_[k] = vn_;
  if (STAGE < 3)
  {
    const T ui = ku * adt_next + ub, vi = kv * adt_next + vb;
    w[k] = ui + s * vi;
    vn[k] = vi;
  }
  else w[k] = un_ + s * vn_;
}

template <typename T>
void launch_stage_westervelt(int stage, bool nl, int64_t n, const void* b, const void* minv, void* u_, void* v_,
                             void* u0, void* v0, void* w, void* vn, double bdt, double adt_next, double s,
                             double kappa, cudaStream_t st)
{
  const unsigned grid = (unsigned)((n + 255) / 256);
#define WFX_STAGE(S, NL)                                                                                    \
  rk_stage_westervelt_kernel<T, S, NL><<<grid, 256, 0, st>>>(n, (const T*)b, (const T*)minv, (T*)u_, (T*)v_, \
                                                              (T*)u0, (T*)v0, (T*)w, (T*)vn, (T)bdt,          \
                                                              (T)adt_next, (T)s, (T)kappa)
  switch (stage * 2 + (nl ? 1 : 0))
  {
  case 0: WFX_STAGE(0, false); break;
  case 1: WFX_STAGE(0, true); break;
  case 2: WFX_STAGE(1, false); break;
  case 3: WFX_STAGE(1, true); break;
  case 4: WFX_STAGE(2, false); break;
  case 5: WFX_STAGE(2, true); break;
  case 6: WFX_STAGE(3, false); break;
  default: WFX_STAGE(3, true); break;
  }
#undef WFX_STAGE
  WFX_CUDA(cudaGetLastError());
}

// w = u + s v: the stiffness input of the lossy / Westervelt models
template <typename T>
__global__ void axpy_kernel(int64_t n, const T* __restrict__ u, const T* __restrict__ v, T s, T* __restrict__ w)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < n) w[k] = u[k] + s * v[k];
}

// f1 of the lossy / Westervelt models: out = (b / m + kappa v^2) / (1 - kappa u), the stage kernel's kv
template <typename T>
__global__ void westervelt_rhs_kernel(int64_t n, const T* __restrict__ b, const T* __restrict__ minv,
                                      const T* __restrict__ u, const T* __restrict__ v, T kappa, T* __restrict__ out)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n) return;
  const T vk = v[k];
  out[k] = (b[k] * minv[k] + kappa * vk * vk) / (T(1) - kappa * u[k]);
}

void launch_axpy(const wfx_wave* w, const void* u, const void* v, double s, void* out, cudaStream_t st)
{
  if (w->n == 0) return;
  const unsigned grid = (unsigned)((w->n + 255) / 256);
  if (w->dtype == WFX_F64)
    axpy_kernel<double><<<grid, 256, 0, st>>>(w->n, (const double*)u, (const double*)v, s, (double*)out);
  else
    axpy_kernel<float><<<grid, 256, 0, st>>>(w->n, (const float*)u, (const float*)v, (float)s, (float*)out);
  WFX_CUDA(cudaGetLastError());
}

// result[i,m] = b[i,m] * minv[i]: the b/m of f1 for an ensemble
template <typename T>
__global__ void scale_rows_kernel(int64_t n, int nv, const T* __restrict__ b, const T* __restrict__ minv,
                                  T* __restrict__ out)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < n * nv) out[k] = b[k] * minv[k / nv];
}

template <typename T>
__global__ void probe_kernel(int64_t n, const int32_t* __restrict__ idx, const T* __restrict__ u, T* __restrict__ out)
{
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = u[idx[i]];
}
// ensemble models: out[p][m] = u[idx[p]][m]
template <typename T>
__global__ void probe_ens_kernel(int64_t n, int nv, const int32_t* __restrict__ idx, const T* __restrict__ u,
                                 T* __restrict__ out)
{
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < n * nv) out[t] = u[(int64_t)idx[t / nv] * nv + t % nv];
}

// Field statistics: e^{-i h w_m t_n} of one sampled step as (cos, -sin) pairs, [h - 1][member], passed by value
struct StatsWeights
{
  double2 e[WFX_HARMONICS_MAX * WFX_ENSEMBLE_MAX];
};
// One sampled step, one thread per entry k (member k % nv, the mapping of rk_stage_ens_kernel): reads u once,
// read-modify-writes the peaks and the nharm fp64 (re, im) pairs, each a coalesced 16-byte access of its plane.
// The pairs are all loaded before any is stored so that their loads are in flight together.
template <typename T>
__global__ void __launch_bounds__(256)
field_stats_kernel(int64_t n, int nv, int nharm, const T* __restrict__ u, T* __restrict__ pmax, T* __restrict__ pmin,
                   double2* __restrict__ harm, const __grid_constant__ StatsWeights wt)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n) return;
  const T x = u[k];
  double2 acc[WFX_HARMONICS_MAX];
#pragma unroll
  for (int h = 0; h < WFX_HARMONICS_MAX; ++h)
    if (h < nharm) acc[h] = harm[h * n + k];
  const T a = pmax[k], b = pmin[k];
  // NaN propagates: a NaN sample replaces the peak, and a NaN peak stays (every comparison with it is false)
  pmax[k] = (x > a || x != x) ? x : a;
  pmin[k] = (x < b || x != x) ? x : b;
  const double xd = (double)x;
  const int m = nv == 1 ? 0 : (int)(k % nv);
#pragma unroll
  for (int h = 0; h < WFX_HARMONICS_MAX; ++h)
    if (h < nharm)
    {
      const double2 e = wt.e[h * WFX_ENSEMBLE_MAX + m];
      acc[h].x = fma(xd, e.x, acc[h].x);
      acc[h].y = fma(xd, e.y, acc[h].y);
      harm[h * n + k] = acc[h];
    }
}

// the statistics' reset state: pmax = -inf, pmin = +inf
template <typename T>
__global__ void fill_peaks_kernel(int64_t n, T* __restrict__ pmax, T* __restrict__ pmin)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < n) pmax[k] = -INFINITY, pmin[k] = INFINITY;
}

// empty accumulators (set_field_stats, init, set_state): ordered after and before all device work, since the
// stepping may run on any of the caller's streams
void reset_field_stats(wfx_wave* w)
{
  w->stats_n = 0;
  w->stats_t_first = w->stats_t_last = 0;
  const int64_t ne = w->n * w->nv;
  if (ne == 0) return;
  WFX_CUDA(cudaDeviceSynchronize());
  const unsigned grid = (unsigned)((ne + 255) / 256);
  if (w->dtype == WFX_F64)
    fill_peaks_kernel<double><<<grid, 256>>>(ne, (double*)w->stats_pmax.p, (double*)w->stats_pmin.p);
  else
    fill_peaks_kernel<float><<<grid, 256>>>(ne, (float*)w->stats_pmax.p, (float*)w->stats_pmin.p);
  WFX_CUDA(cudaGetLastError());
  if (w->stats_nharm) WFX_CUDA(cudaMemsetAsync(w->stats_harm.p, 0, w->stats_harm.n * sizeof(double2), nullptr));
  WFX_CUDA(cudaDeviceSynchronize());
}

// one sampled step at the time reached, w->t_now
void sample_field_stats(wfx_wave* w, cudaStream_t ws)
{
  const double t = w->t_now;
  if (w->stats_n == 0) w->stats_t_first = t;
  w->stats_t_last = t;
  w->stats_n += 1;
  const int64_t ne = w->n * w->nv;
  if (ne == 0) return;
  StatsWeights wt{};
  for (int h = 1; h <= w->stats_nharm; ++h)
    for (int m = 0; m < w->nv; ++m)
    {
      const double w0 = 2.0 * M_PI * (w->ens ? w->f0s[m] : w->f0);
      const double ph = h * w0 * t;
      wt.e[(h - 1) * WFX_ENSEMBLE_MAX + m] = make_double2(std::cos(ph), -std::sin(ph));
    }
  const unsigned grid = (unsigned)((ne + 255) / 256);
  if (w->dtype == WFX_F64)
    field_stats_kernel<double><<<grid, 256, 0, ws>>>(ne, w->nv, w->stats_nharm, (const double*)w->u_.p,
                                                      (double*)w->stats_pmax.p, (double*)w->stats_pmin.p,
                                                      w->stats_harm.p, wt);
  else
    field_stats_kernel<float><<<grid, 256, 0, ws>>>(ne, w->nv, w->stats_nharm, (const float*)w->u_.p,
                                                     (float*)w->stats_pmax.p, (float*)w->stats_pmin.p,
                                                     w->stats_harm.p, wt);
  WFX_CUDA(cudaGetLastError());
}

// the pending snapshot's copy has landed: hand it to the callback
void flush_snapshot(wfx_wave* w)
{
  if (!w->snap_pending) return;
  WFX_CUDA(cudaEventSynchronize(w->ev_snap_done));
  w->snap_pending = false;
  if (w->snap_fn) w->snap_fn(w->snap_user, w->snap_step, w->snap_t, w->snap_hu, w->snap_hv);
}

// after a completed step of size dt: probe record, field statistics inside their window and, every snap_every
// steps, a snapshot.  The half step in the window test keeps rounding in the accumulated t from moving its edge.
void after_step(wfx_wave* w, double dt, cudaStream_t ws)
{
  const size_t esz = w->dtype == WFX_F64 ? 8 : 4;
  if (w->stats_on && w->t_now >= w->stats_t_start - 0.5 * dt) sample_field_stats(w, ws);
  if (w->nprobes && w->probe_rec < w->probe_cap)
  {
    const unsigned grid = (unsigned)((w->nprobes * w->nv + 255) / 256);
    unsigned char* out = w->d_probe_val.p + (size_t)w->probe_rec * w->nprobes * w->nv * esz;
    if (w->ens && w->dtype == WFX_F64)
      probe_ens_kernel<double><<<grid, 256, 0, ws>>>(w->nprobes, w->nv, w->d_probe_idx.p, (const double*)w->u_.p, (double*)out);
    else if (w->ens)
      probe_ens_kernel<float><<<grid, 256, 0, ws>>>(w->nprobes, w->nv, w->d_probe_idx.p, (const float*)w->u_.p, (float*)out);
    else if (w->dtype == WFX_F64)
      probe_kernel<double><<<grid, 256, 0, ws>>>(w->nprobes, w->d_probe_idx.p, (const double*)w->u_.p, (double*)out);
    else
      probe_kernel<float><<<grid, 256, 0, ws>>>(w->nprobes, w->d_probe_idx.p, (const float*)w->u_.p, (float*)out);
    WFX_CUDA(cudaGetLastError());
    w->probe_t.push_back(w->t_now);
    w->probe_rec += 1;
  }
  if (w->snap_every > 0 && w->steps_done % w->snap_every == 0)
  {
    flush_snapshot(w); // the staging buffers are free again (usually long since)
    const size_t nb = (size_t)w->n * esz;
    WFX_CUDA(cudaMemcpyAsync(w->snap_u.p, w->u_.p, nb, cudaMemcpyDeviceToDevice, ws));
    WFX_CUDA(cudaMemcpyAsync(w->snap_v.p, w->v_.p, nb, cudaMemcpyDeviceToDevice, ws));
    WFX_CUDA(cudaEventRecord(w->ev_snap_ready, ws));
    WFX_CUDA(cudaStreamWaitEvent(w->snap_stream, w->ev_snap_ready, 0));
    WFX_CUDA(cudaMemcpyAsync(w->snap_hu, w->snap_u.p, nb, cudaMemcpyDeviceToHost, w->snap_stream));
    WFX_CUDA(cudaMemcpyAsync(w->snap_hv, w->snap_v.p, nb, cudaMemcpyDeviceToHost, w->snap_stream));
    WFX_CUDA(cudaEventRecord(w->ev_snap_done, w->snap_stream));
    // the next snapshot's device copy must not overtake this one's read: ws waits for it then
    w->snap_pending = true;
    w->snap_step = w->steps_done;
    w->snap_t = w->t_now;
  }
}

__global__ void set_source_kernel(double* g_dev, double g0, double g1, double g2, double g3)
{
  g_dev[0] = g0, g_dev[1] = g1, g_dev[2] = g2, g_dev[3] = g3;
}
// ensemble models: the 4 x nv amplitudes of a step, [stage][member], passed by value
struct StepAmp
{
  double g[4 * WFX_ENSEMBLE_MAX];
};
__global__ void set_source_ens_kernel(double* g_dev, const StepAmp a, int n)
{
  if ((int)threadIdx.x < n) g_dev[threadIdx.x] = a.g[threadIdx.x];
}

void boundary_profiled(wfx_wave* w, double tn, const double* t_dev, const void* vn, cudaStream_t st);

// One time step of size dt on stream st: the four stages of LinearGLL.hpp:244-270.  g[i*nv + m] is the
// source amplitude of stage i (of member m); with g_from_dev the boundary kernels read it from w->g_dev
// instead (graph capture).  With a source profile the boundary term takes the stage times tn[i] instead, or
// reads them from w->t_dev.
void enqueue_step(wfx_wave* w, double dt, const double* g, const double* tn, bool g_from_dev, cudaStream_t st)
{
  const double a_runge[5] = {0.0, 0.5, 0.5, 1.0, 0.0};
  const double b_runge[4] = {1.0 / 6.0, 1.0 / 3.0, 1.0 / 3.0, 1.0 / 6.0};
  auto boundary = [&](int i, const void* vn) {
    if (!w->bnd) return;
    if (w->prof_on) boundary_profiled(w, g_from_dev ? 0.0 : tn[i], g_from_dev ? w->t_dev.p + i : nullptr, vn, st);
    else if (w->ens)
      boundary_apply_ens(w->bnd, w->nv, w->c0, g_from_dev ? nullptr : g + i * w->nv,
                         g_from_dev ? w->g_dev.p + i * w->nv : nullptr, vn, w->b.p, st);
    else if (g_from_dev) boundary_apply_dev(w->bnd, w->c0, w->g_dev.p + i, vn, w->b.p, st);
    else if (wfx_boundary_apply(w->bnd, w->c0, g[i], vn, w->b.p, st)) fail("%s", wfx_last_error()); // :175
  };
  static const char* const stage_name[4] = {"wfx rk4 stage 0", "wfx rk4 stage 1", "wfx rk4 stage 2", "wfx rk4 stage 3"};
  for (int i = 0; i < 4; ++i)
  {
    NvtxRange stage_range(stage_name[i]);
    // stage state: the solution itself at stage 0 (a_0 = 0), else un/vn.  Lossy / Westervelt models:
    // the stiffness input is w = un + s vn, kept in `un` at every stage
    const void* un = i == 0 && !w->model ? w->u_.p : w->un.p;
    const void* vn = i == 0 ? w->v_.p : w->vn.p;
    // f1 (:151-192)
    if (!w->halo)
    {
      {
        NvtxRange r("wfx stiffness apply");
        const int rc = w->ens ? wfx_stiffness_apply_ensemble(w->stiff, w->nv, un, nullptr, w->b.p, 0, st)
                              : wfx_stiffness_apply(w->stiff, un, w->b.p, 0, st); // :173-174
        if (rc) fail("%s", wfx_last_error());
      }
      boundary(i, vn);
    }
    else
    {
      // distributed: interface cells first, their ghost reduction (:176, which also stands
      // for the scatter_fwd of the next stage, :164,167) on the comm stream while the interior
      // cells run; the boundary term (facet masses assembled over the ranks) is added by
      // every copy of a dof after the reduction.
      static const bool overlap = [] { const char* e = std::getenv("WFX_WAVE_OVERLAP"); return !e || std::atoi(e) != 0; }();
      const bool split = overlap && stiffness_has_split(w->stiff);
      {
        NvtxRange r("wfx stiffness interface part");
        if (wfx_stiffness_apply_part(w->stiff, un, nullptr, w->b.p, 0, split ? 0 : -1, st)) fail("%s", wfx_last_error());
      }
      WFX_CUDA(cudaEventRecord(w->ev_iface, st));
      WFX_CUDA(cudaStreamWaitEvent(w->comm_stream, w->ev_iface, 0));
      {
        NvtxRange r("wfx ghost reduction");
        if (wfx_halo_update_rev_fwd(w->halo, w->b.p, w->comm_stream)) fail("%s", wfx_last_error());
      }
      WFX_CUDA(cudaEventRecord(w->ev_halo, w->comm_stream));
      {
        NvtxRange r("wfx stiffness interior part");
        if (split && wfx_stiffness_apply_part(w->stiff, un, nullptr, w->b.p, 0, 1, st)) fail("%s", wfx_last_error());
      }
      WFX_CUDA(cudaStreamWaitEvent(st, w->ev_halo, 0));
      boundary(i, vn);
    }
    if (w->model)
    {
      // Gamma2 mass term (compact, absorbing dofs), then the fused update; p = u_ at stage 0, else w - s vn
      if (w->qc != 0)
        boundary_absorbing_mass(w->bnd, w->m64, w->qc, w->kappa, i == 0 ? 0.0 : w->s_stiff,
                                i == 0 ? w->u_.p : w->un.p, vn, w->b.p, st);
      NvtxRange update_range("wfx fused stage update");
      if (w->dtype == WFX_F64)
        launch_stage_westervelt<double>(i, w->model == 2, w->n, w->b.p, w->minv, w->u_.p, w->v_.p, w->u0.p, w->v0.p,
                                        w->un.p, w->vn.p, dt * b_runge[i], dt * a_runge[i + 1], w->s_stiff, w->kappa, st);
      else
        launch_stage_westervelt<float>(i, w->model == 2, w->n, w->b.p, w->minv, w->u_.p, w->v_.p, w->u0.p, w->v0.p,
                                       w->un.p, w->vn.p, dt * b_runge[i], dt * a_runge[i + 1], w->s_stiff, w->kappa, st);
      continue;
    }
    NvtxRange update_range("wfx fused stage update");
    if (w->ens && w->dtype == WFX_F64)
      launch_stage_ens<double>(i, w->n, w->nv, w->b.p, w->minv, w->u_.p, w->v_.p, w->u0.p, w->v0.p, w->un.p,
                               w->vn.p, dt * b_runge[i], dt * a_runge[i + 1], st);
    else if (w->ens)
      launch_stage_ens<float>(i, w->n, w->nv, w->b.p, w->minv, w->u_.p, w->v_.p, w->u0.p, w->v0.p, w->un.p,
                              w->vn.p, dt * b_runge[i], dt * a_runge[i + 1], st);
    else if (w->dtype == WFX_F64)
      launch_stage<double>(i, w->n, w->b.p, w->minv, w->u_.p, w->v_.p, w->u0.p, w->v0.p, w->un.p,
                           w->vn.p, dt * b_runge[i], dt * a_runge[i + 1], st);
    else
      launch_stage<float>(i, w->n, w->b.p, w->minv, w->u_.p, w->v_.p, w->u0.p, w->v0.p, w->un.p,
                          w->vn.p, dt * b_runge[i], dt * a_runge[i + 1], st);
  }
}
} // namespace

extern "C" int wfx_wave_create(wfx_ctx* ctx, wfx_stiffness* stiff, wfx_mass* mass,
                               wfx_boundary* bnd, wfx_halo* halo, int64_t size_local, double c0,
                               double f0, double p0, wfx_wave** out)
{
  WFX_API_BEGIN
  if (!ctx || !stiff || !mass || !out) fail("NULL argument");
  ScopedDevice sd(ctx->device);
  int64_t ndofs = 0;
  if (wfx_stiffness_info(stiff, nullptr, nullptr, &ndofs, nullptr, nullptr, nullptr, nullptr))
    fail("%s", wfx_last_error());
  auto w = std::make_unique<wfx_wave>();
  w->ctx = ctx;
  w->stiff = stiff;
  w->mass = mass;
  w->bnd = bnd;
  w->halo = halo;
  w->n = ndofs;
  w->size_local = size_local;
  w->c0 = c0;
  w->f0 = f0;
  w->p0 = p0;
  w->dtype = stiffness_dtype(stiff);
  if (mass_dtype(mass) != w->dtype) fail("wave: mass operator dtype differs from the stiffness operator's");
  if (bnd && boundary_dtype(bnd) != w->dtype) fail("wave: boundary operator dtype differs from the stiffness operator's");
  if (halo)
  {
    // every stage exchanges the model's right-hand side through this halo: same scalar type or
    // the buffers are reinterpreted
    if (halo_dtype(halo) != w->dtype) fail("wave: halo dtype differs from the model dtype");
    // m.scatter_rev(add) (LinearGLL.hpp:110) and the same for the facet masses (both idempotent).
    // They are summed in fp64: an fp64 model's halo serves, an fp32 model must have assembled them
    // beforehand with a separate fp64 halo (wfx_mass_assemble / wfx_boundary_assemble).
    if (w->dtype == WFX_F64)
    {
      if (wfx_mass_assemble(mass, halo)) fail("%s", wfx_last_error());
      if (bnd && wfx_boundary_assemble(bnd, halo)) fail("%s", wfx_last_error());
    }
    if (!mass_assembled(mass))
      fail("wave: distributed fp32 model needs the mass assembled first (wfx_mass_assemble with an fp64 halo)");
    if (bnd && !boundary_assembled(bnd))
      fail("wave: distributed fp32 model needs the facet masses assembled first (wfx_boundary_assemble with an fp64 halo)");
    // highest priority: the small pack / NCCL / unpack kernels must not queue behind the interior batches
    int prio_lo = 0, prio_hi = 0;
    WFX_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    WFX_CUDA(cudaStreamCreateWithPriority(&w->comm_stream, cudaStreamNonBlocking, prio_hi));
    WFX_CUDA(cudaEventCreateWithFlags(&w->ev_iface, cudaEventDisableTiming));
    WFX_CUDA(cudaEventCreateWithFlags(&w->ev_halo, cudaEventDisableTiming));
  }
  if (const char* e = std::getenv("WFX_WAVE_GRAPH")) w->use_graph = std::atoi(e) != 0;
  if (!halo)
  {
    w->g_dev.alloc(4);
    w->t_dev.alloc(4);
    WFX_CUDA(cudaStreamCreateWithFlags(&w->own_stream, cudaStreamNonBlocking));
    WFX_CUDA(cudaEventCreateWithFlags(&w->ev_in, cudaEventDisableTiming));
    WFX_CUDA(cudaEventCreateWithFlags(&w->ev_out, cudaEventDisableTiming));
  }
  if (wfx_mass_inverse_diagonal(mass, &w->minv)) fail("%s", wfx_last_error());
  const size_t nb = (size_t)ndofs * (w->dtype == WFX_F64 ? 8 : 4);
  for (auto* v : {&w->u_, &w->v_, &w->u0, &w->v0, &w->un, &w->vn, &w->b})
  {
    v->alloc(nb);
    if (nb) WFX_CUDA(cudaMemset(v->p, 0, nb));
  }
  *out = w.release();
  WFX_API_END
}

extern "C" int wfx_wave_create_ensemble(wfx_ctx* ctx, wfx_stiffness* stiff, wfx_mass* mass, wfx_boundary* bnd,
                                        int nv, int64_t size_local, double c0, const double* f0_host,
                                        const double* p0_host, wfx_wave** out)
{
  WFX_API_BEGIN
  if (!ctx || !stiff || !mass || !out || !f0_host || !p0_host) fail("NULL argument");
  if (nv < 1 || nv > WFX_ENSEMBLE_MAX) fail("wave ensemble: nv = %d outside [1, %d]", nv, WFX_ENSEMBLE_MAX);
  if (!stiffness_has_ensemble(stiff))
    fail("wave ensemble: the stiffness operator needs WFX_STIFF_ENSEMBLE and no rank-shared dofs");
  for (int m = 0; m < nv; ++m)
    if (!(f0_host[m] > 0)) fail("wave ensemble: source frequency of member %d must be positive", m);
  wfx_wave* w = nullptr;
  if (wfx_wave_create(ctx, stiff, mass, bnd, nullptr, size_local, c0, f0_host[0], p0_host[0], &w))
    fail("%s", wfx_last_error());
  std::unique_ptr<wfx_wave> guard(w);
  ScopedDevice sd(ctx->device);
  w->ens = true;
  w->nv = nv;
  w->f0s.assign(f0_host, f0_host + nv);
  w->p0s.assign(p0_host, p0_host + nv);
  w->g_dev.alloc(4 * WFX_ENSEMBLE_MAX);
  const size_t nb = (size_t)w->n * nv * (w->dtype == WFX_F64 ? 8 : 4);
  for (auto* v : {&w->u_, &w->v_, &w->u0, &w->v0, &w->un, &w->vn, &w->b})
  {
    v->alloc(nb);
    if (nb) WFX_CUDA(cudaMemset(v->p, 0, nb));
  }
  *out = guard.release();
  WFX_API_END
}

extern "C" int wfx_wave_create_westervelt(wfx_ctx* ctx, wfx_stiffness* stiff, wfx_mass* mass, wfx_boundary* bnd,
                                          int64_t size_local, double c0, double f0, double p0, double delta,
                                          double beta, double rho0, wfx_wave** out)
{
  WFX_API_BEGIN
  if (!ctx || !stiff || !mass || !out) fail("NULL argument");
  for (double x : {c0, f0, p0, delta, beta, rho0})
    if (!std::isfinite(x)) fail("wave westervelt: non-finite parameter");
  if (!(c0 > 0)) fail("wave westervelt: speed of sound must be positive");
  if (!(f0 > 0)) fail("wave westervelt: source frequency must be positive");
  if (delta < 0) fail("wave westervelt: diffusivity of sound delta must not be negative");
  if (beta < 0) fail("wave westervelt: coefficient of nonlinearity beta must not be negative");
  if (beta > 0 && !(rho0 > 0)) fail("wave westervelt: density rho0 must be positive when beta > 0");
  if (stiffness_nshared(stiff) > 0) fail("wave westervelt: one rank only (the stiffness operator has rank-shared dofs)");
  wfx_wave* w = nullptr;
  if (wfx_wave_create(ctx, stiff, mass, bnd, nullptr, size_local, c0, f0, p0, &w)) fail("%s", wfx_last_error());
  std::unique_ptr<wfx_wave> guard(w);
  w->model = beta > 0 ? 2 : 1;
  w->kappa = beta > 0 ? 2.0 * beta / (rho0 * c0 * c0) : 0.0;
  // -delta K v = (delta / cK^2) (-cK^2 K v) with cK the operator's c0; c0^2 (g + s_src g') = c0^2 g + delta g'
  const double cK = stiffness_c0(stiff);
  w->s_stiff = delta / (cK * cK);
  w->s_src = delta / (c0 * c0);
  w->qc = bnd ? delta / c0 : 0.0;
  w->m64 = mass_diagonal64(mass);
  *out = guard.release();
  WFX_API_END
}

extern "C" int wfx_wave_init(wfx_wave* w)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  ScopedDevice sd(w->ctx->device);
  if (w->u_.n)
  {
    WFX_CUDA(cudaMemset(w->u_.p, 0, w->u_.n));
    WFX_CUDA(cudaMemset(w->v_.p, 0, w->v_.n));
  }
  w->steps_done = 0;
  w->t_now = 0;
  w->probe_rec = 0;
  w->probe_t.clear();
  if (w->stats_on) reset_field_stats(w);
  WFX_API_END
}

extern "C" int wfx_wave_set_state(wfx_wave* w, const void* u, const void* v)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  ScopedDevice sd(w->ctx->device);
  if (u && w->u_.n) WFX_CUDA(cudaMemcpy(w->u_.p, u, w->u_.n, cudaMemcpyHostToDevice));
  if (v && w->v_.n) WFX_CUDA(cudaMemcpy(w->v_.p, v, w->v_.n, cudaMemcpyHostToDevice));
  w->steps_done = 0;
  w->t_now = 0;
  w->probe_rec = 0;
  w->probe_t.clear();
  if (w->stats_on) reset_field_stats(w);
  // u->scatter_fwd(), v->scatter_fwd() (LinearGLL.hpp:164,167): the stage kernels update ghost
  // entries locally from then on, so the copies are made consistent once, here
  if (w->halo && w->n)
  {
    if (u && wfx_halo_update_fwd(w->halo, w->u_.p, nullptr)) fail("%s", wfx_last_error());
    if (v && wfx_halo_update_fwd(w->halo, w->v_.p, nullptr)) fail("%s", wfx_last_error());
    WFX_CUDA(cudaDeviceSynchronize());
  }
  WFX_API_END
}

extern "C" int wfx_wave_get_state(wfx_wave* w, void* u, void* v)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  ScopedDevice sd(w->ctx->device);
  if (u && w->u_.n) WFX_CUDA(cudaMemcpy(u, w->u_.p, w->u_.n, cudaMemcpyDeviceToHost));
  if (v && w->v_.n) WFX_CUDA(cudaMemcpy(v, w->v_.p, w->v_.n, cudaMemcpyDeviceToHost));
  WFX_API_END
}

extern "C" int wfx_wave_state_ptrs(wfx_wave* w, void** u, void** v)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  if (u) *u = w->u_.p;
  if (v) *v = w->v_.p;
  WFX_API_END
}

namespace
{
// g(t) of LinearGLL.hpp:155-162 (source_eval, wfx_source.h)
double source_amplitude(double f0, double p0, double c0, double tn)
{
  double g, gdot;
  source_eval(f0, p0, c0, tn, &g, &gdot);
  return g;
}
// the amplitude the boundary term receives: g, or g + (delta / c0^2) g' for the lossy / Westervelt models
double source_amplitude(const wfx_wave* w, double tn)
{
  double g, gdot;
  source_eval(w->f0, w->p0, w->c0, tn, &g, &gdot);
  return w->model ? g + w->s_src * gdot : g;
}
// g_m(t) of every member (ensemble models): g[m], m < nv
void source_amplitudes(const wfx_wave* w, double tn, double* g)
{
  for (int m = 0; m < w->nv; ++m) g[m] = source_amplitude(w->f0s[m], w->p0s[m], w->c0, tn);
}
// the boundary term with the source profile at stage time tn (t_dev: read it from there, graph capture)
void boundary_profiled(wfx_wave* w, double tn, const double* t_dev, const void* vn, cudaStream_t st)
{
  SourceParams sp{};
  for (int m = 0; m < w->nv; ++m)
  {
    sp.f0[m] = w->ens ? w->f0s[m] : w->f0;
    sp.p0[m] = w->ens ? w->p0s[m] : w->p0;
  }
  boundary_apply_profile(w->bnd, w->nv, w->c0, w->model ? w->s_src : 0.0, sp, tn, t_dev, w->prof_amp.p,
                         w->prof_delay.p, vn, w->b.p, st);
}
} // namespace

extern "C" int wfx_wave_f0(wfx_wave* w, double, const void* u, const void* v, void* result, void* stream)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  if (!u || !v || !result) fail("f0: NULL vector");
  ScopedDevice sd(w->ctx->device);
  const size_t nb = (size_t)w->n * w->nv * (w->dtype == WFX_F64 ? 8 : 4);
  if (result != v) WFX_CUDA(cudaMemcpyAsync(result, v, nb, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  WFX_API_END
}

extern "C" int wfx_wave_f1(wfx_wave* w, double t, const void* u, const void* v, void* result, void* stream)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  if (!u || !v || !result) fail("f1: NULL vector");
  if (result == u || result == v) fail("f1: result must not alias u or v");
  ScopedDevice sd(w->ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (w->ens)
  {
    double g[WFX_ENSEMBLE_MAX];
    source_amplitudes(w, t, g);
    if (wfx_stiffness_apply_ensemble(w->stiff, w->nv, u, nullptr, w->b.p, 0, st)) fail("%s", wfx_last_error());
    if (w->prof_on) boundary_profiled(w, t, nullptr, v, st);
    else boundary_apply_ens(w->bnd, w->nv, w->c0, g, nullptr, v, w->b.p, st);
    const int64_t n = w->n * w->nv;
    if (n == 0) return 0;
    const unsigned grid = (unsigned)((n + 255) / 256);
    if (w->dtype == WFX_F64)
      scale_rows_kernel<double><<<grid, 256, 0, st>>>(w->n, w->nv, (const double*)w->b.p, (const double*)w->minv, (double*)result);
    else
      scale_rows_kernel<float><<<grid, 256, 0, st>>>(w->n, w->nv, (const float*)w->b.p, (const float*)w->minv, (float*)result);
    WFX_CUDA(cudaGetLastError());
    return 0;
  }
  const double g = source_amplitude(w, t);
  if (w->model)
  {
    // w = u + s v in a scratch vector of its own (the rk4 one carries the state of the next step)
    const size_t nb = (size_t)w->n * (w->dtype == WFX_F64 ? 8 : 4);
    if (w->f1_w.n != nb) w->f1_w.alloc(nb);
    launch_axpy(w, u, v, w->s_stiff, w->f1_w.p, st);
    if (wfx_stiffness_apply(w->stiff, w->f1_w.p, w->b.p, 0, st)) fail("%s", wfx_last_error());
    if (w->prof_on) boundary_profiled(w, t, nullptr, v, st);
    else if (w->bnd && wfx_boundary_apply(w->bnd, w->c0, g, v, w->b.p, st)) fail("%s", wfx_last_error());
    if (w->qc != 0) boundary_absorbing_mass(w->bnd, w->m64, w->qc, w->kappa, 0.0, u, v, w->b.p, st);
    if (w->n == 0) return 0;
    const unsigned grid = (unsigned)((w->n + 255) / 256);
    if (w->dtype == WFX_F64)
      westervelt_rhs_kernel<double><<<grid, 256, 0, st>>>(w->n, (const double*)w->b.p, (const double*)w->minv,
                                                           (const double*)u, (const double*)v, w->kappa, (double*)result);
    else
      westervelt_rhs_kernel<float><<<grid, 256, 0, st>>>(w->n, (const float*)w->b.p, (const float*)w->minv,
                                                          (const float*)u, (const float*)v, (float)w->kappa, (float*)result);
    WFX_CUDA(cudaGetLastError());
    return 0;
  }
  if (wfx_stiffness_apply(w->stiff, u, w->b.p, 0, st)) fail("%s", wfx_last_error());                     // :173-174
  if (w->halo && wfx_halo_update_rev_fwd(w->halo, w->b.p, st)) fail("%s", wfx_last_error());             // :176
  if (w->prof_on) boundary_profiled(w, t, nullptr, v, st);
  else if (w->bnd && wfx_boundary_apply(w->bnd, w->c0, g, v, w->b.p, st)) fail("%s", wfx_last_error());  // :175
  if (wfx_mass_apply_inverse(w->mass, w->b.p, result, st)) fail("%s", wfx_last_error());                 // :188-191
  WFX_API_END
}

extern "C" int wfx_wave_rk4(wfx_wave* w, double t0, double tf, double dt, int64_t max_steps,
                            int64_t* steps_out, double* t_end, void* stream)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  ScopedDevice sd(w->ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  const double c_runge[4] = {0.0, 0.5, 0.5, 1.0};
  // Graph replay (one rank only: the distributed step spans two streams and NCCL).  A capture
  // cannot run on the legacy default stream: such callers are moved to an internal stream that
  // is ordered after and before the caller's stream by events.
  const bool graph_ok = w->use_graph && !w->halo && stiffness_graph_safe(w->stiff);
  cudaStream_t ws = st;
  if (graph_ok && (st == nullptr || st == cudaStreamLegacy))
  {
    ws = w->own_stream;
    WFX_CUDA(cudaEventRecord(w->ev_in, st));
    WFX_CUDA(cudaStreamWaitEvent(ws, w->ev_in, 0));
  }
  // lossy / Westervelt models: the stiffness input w = u_ + s v_ of the first stage, rebuilt on every call so
  // that it follows init, set_state, a restart or writes through wfx_wave_state_ptrs (later steps get it
  // from stage 3 of the step before)
  if (w->model) launch_axpy(w, w->u_.p, w->v_.p, w->s_stiff, w->un.p, ws);
  double t = t0;
  int64_t step = 0;
  const double dt_nominal = dt;
  while (t < tf) // :241
  {
    if (max_steps > 0 && step >= max_steps) break;
    NvtxRange step_range("wfx rk4 step");
    dt = std::min(dt, tf - t); // :242
    double g[4 * WFX_ENSEMBLE_MAX]; // [stage][member]
    double tn[4];
    for (int i = 0; i < 4; ++i)
    {
      tn[i] = t + c_runge[i] * dt; // :257
      if (w->prof_on) continue;    // the boundary term evaluates the delayed sources on the device
      if (w->ens) source_amplitudes(w, tn[i], g + i * w->nv);
      else g[i] = source_amplitude(w, tn[i]); // :155-162
    }
    if (graph_ok && dt == dt_nominal)
    {
      if (!w->step_graph || w->graph_dt != dt)
      {
        if (w->step_graph) WFX_CUDA(cudaGraphExecDestroy(w->step_graph));
        w->step_graph = nullptr;
        cudaGraph_t graph = nullptr;
        WFX_CUDA(cudaStreamBeginCapture(ws, cudaStreamCaptureModeThreadLocal));
        try
        {
          enqueue_step(w, dt, nullptr, nullptr, true, ws);
        }
        catch (...)
        {
          cudaStreamEndCapture(ws, &graph);
          if (graph) cudaGraphDestroy(graph);
          throw;
        }
        WFX_CUDA(cudaStreamEndCapture(ws, &graph));
        const cudaError_t ie = cudaGraphInstantiate(&w->step_graph, graph, 0);
        cudaGraphDestroy(graph);
        WFX_CUDA(ie);
        w->graph_dt = dt;
      }
      if (w->prof_on) set_source_kernel<<<1, 1, 0, ws>>>(w->t_dev.p, tn[0], tn[1], tn[2], tn[3]);
      else if (w->ens)
      {
        StepAmp a{};
        for (int q = 0; q < 4 * w->nv; ++q) a.g[q] = g[q];
        set_source_ens_kernel<<<1, 4 * WFX_ENSEMBLE_MAX, 0, ws>>>(w->g_dev.p, a, 4 * w->nv);
      }
      else set_source_kernel<<<1, 1, 0, ws>>>(w->g_dev.p, g[0], g[1], g[2], g[3]);
      WFX_CUDA(cudaGraphLaunch(w->step_graph, ws));
    }
    else enqueue_step(w, dt, g, tn, false, ws);
    t += dt;
    step += 1;
    w->steps_done += 1;
    w->t_now = t;
    if (w->nprobes || w->snap_every > 0 || w->stats_on)
    {
      if (w->snap_pending && w->snap_every > 0 && (w->steps_done % w->snap_every) == 0)
        WFX_CUDA(cudaStreamWaitEvent(ws, w->ev_snap_done, 0));
      after_step(w, dt, ws);
    }
  }
  if (w->snap_pending)
  {
    // deliver the last snapshot before returning (the callback may read solver state)
    flush_snapshot(w);
  }
  if (ws != st)
  {
    WFX_CUDA(cudaEventRecord(w->ev_out, ws));
    WFX_CUDA(cudaStreamWaitEvent(st, w->ev_out, 0));
  }
  if (steps_out) *steps_out = step;
  if (t_end) *t_end = t;
  WFX_API_END
}

extern "C" int wfx_wave_set_probes(wfx_wave* w, int64_t nprobes, const int32_t* dofs_host, int64_t max_records)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  if (nprobes < 0 || max_records < 0 || (nprobes > 0 && !dofs_host)) fail("bad probe list");
  for (int64_t i = 0; i < nprobes; ++i)
    if (dofs_host[i] < 0 || dofs_host[i] >= w->n) fail("probe dof %d out of range", dofs_host[i]);
  ScopedDevice sd(w->ctx->device);
  w->nprobes = nprobes;
  w->probe_cap = nprobes ? max_records : 0;
  w->probe_rec = 0;
  w->probe_t.clear();
  if (nprobes)
  {
    w->d_probe_idx.upload(dofs_host, (size_t)nprobes);
    w->d_probe_val.alloc((size_t)nprobes * (size_t)max_records * w->nv * (w->dtype == WFX_F64 ? 8 : 4));
  }
  WFX_API_END
}

extern "C" int wfx_wave_get_probe_series(wfx_wave* w, int64_t* nrecords, double* t_host, void* values_host)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  ScopedDevice sd(w->ctx->device);
  if (nrecords) *nrecords = w->probe_rec;
  if (t_host)
    for (int64_t r = 0; r < w->probe_rec; ++r) t_host[r] = w->probe_t[r];
  if (values_host && w->probe_rec)
  {
    WFX_CUDA(cudaDeviceSynchronize());
    WFX_CUDA(cudaMemcpy(values_host, w->d_probe_val.p,
                        (size_t)w->probe_rec * w->nprobes * w->nv * (w->dtype == WFX_F64 ? 8 : 4), cudaMemcpyDeviceToHost));
  }
  WFX_API_END
}

extern "C" int wfx_wave_set_field_stats(wfx_wave* w, int enable, double t_start, int nharm)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  if (enable && (nharm < 0 || nharm > WFX_HARMONICS_MAX))
    fail("field statistics: nharm = %d outside [0, %d]", nharm, WFX_HARMONICS_MAX);
  if (enable && !std::isfinite(t_start)) fail("field statistics: t_start must be finite");
  ScopedDevice sd(w->ctx->device);
  WFX_CUDA(cudaDeviceSynchronize()); // the buffers may still be in use by a step in flight
  w->stats_on = false;
  w->stats_n = 0;
  if (!enable)
  {
    w->stats_nharm = 0;
    w->stats_pmax.release();
    w->stats_pmin.release();
    w->stats_harm.release();
    return 0;
  }
  const size_t ne = (size_t)w->n * w->nv, nb = ne * (w->dtype == WFX_F64 ? 8 : 4);
  // each buffer on its own: after a failed allocation (out of memory) a retry allocates what is missing
  if (w->stats_pmax.n != nb) w->stats_pmax.alloc(nb);
  if (w->stats_pmin.n != nb) w->stats_pmin.alloc(nb);
  if (w->stats_harm.n != ne * nharm) w->stats_harm.alloc(ne * nharm);
  w->stats_nharm = nharm;
  w->stats_t_start = t_start;
  w->stats_on = true;
  reset_field_stats(w);
  WFX_API_END
}

extern "C" int wfx_wave_field_stats_info(wfx_wave* w, int* enabled, double* t_start, int* nharm)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  if (enabled) *enabled = w->stats_on ? 1 : 0;
  if (t_start) *t_start = w->stats_on ? w->stats_t_start : 0.0;
  if (nharm) *nharm = w->stats_on ? w->stats_nharm : 0;
  WFX_API_END
}

extern "C" int wfx_wave_get_field_stats(wfx_wave* w, int64_t* nsamples, double* t_first, double* t_last,
                                        void* pmax_host, void* pmin_host, double* harm_host)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  if (!w->stats_on) fail("field statistics are off (wfx_wave_set_field_stats)");
  ScopedDevice sd(w->ctx->device);
  if (nsamples) *nsamples = w->stats_n;
  if (t_first) *t_first = w->stats_t_first;
  if (t_last) *t_last = w->stats_t_last;
  if (!pmax_host && !pmin_host && !harm_host) return 0;
  WFX_CUDA(cudaDeviceSynchronize());
  if (pmax_host) w->stats_pmax.download((unsigned char*)pmax_host, w->stats_pmax.n);
  if (pmin_host) w->stats_pmin.download((unsigned char*)pmin_host, w->stats_pmin.n);
  if (harm_host && w->stats_harm.n)
  {
    w->stats_harm.download((double2*)harm_host, w->stats_harm.n);
    const double scale = w->stats_n ? 2.0 / (double)w->stats_n : 0.0;
    for (size_t i = 0; i < 2 * w->stats_harm.n; ++i) harm_host[i] *= scale;
  }
  WFX_API_END
}

WaveFieldStats wfx::wave_field_stats(const wfx_wave* w)
{
  WaveFieldStats s;
  s.ctx = w->ctx;
  s.ndofs = w->n;
  s.nv = w->nv;
  s.on = w->stats_on;
  s.nharm = w->stats_on ? w->stats_nharm : 0;
  s.nsamples = w->stats_n;
  s.harm = w->stats_harm.p;
  for (int m = 0; m < w->nv; ++m) s.f0[m] = w->ens ? w->f0s[m] : w->f0;
  return s;
}

extern "C" int wfx_wave_set_source_profile(wfx_wave* w, const double* amp_host, const double* delay_host)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  if (!w->bnd) fail("source profile: the model has no boundary operator");
  if (w->halo) fail("source profile: one rank only (the model is distributed)");
  const int64_t ne = w->n * w->nv;
  for (int64_t k = 0; k < ne; ++k)
  {
    if (amp_host && !std::isfinite(amp_host[k])) fail("source profile: non-finite amplitude at entry %lld", (long long)k);
    if (delay_host && !std::isfinite(delay_host[k])) fail("source profile: non-finite delay at entry %lld", (long long)k);
    if (delay_host && delay_host[k] < 0) fail("source profile: negative delay at entry %lld", (long long)k);
  }
  ScopedDevice sd(w->ctx->device);
  // a step in flight may read the buffers, and the captured step holds the other boundary kernel (or these buffers)
  WFX_CUDA(cudaDeviceSynchronize());
  if (w->step_graph) WFX_CUDA(cudaGraphExecDestroy(w->step_graph));
  w->step_graph = nullptr;
  w->prof_on = false;
  if (!amp_host && !delay_host)
  {
    w->prof_amp.release();
    w->prof_delay.release();
    return 0;
  }
  // compact onto the boundary term's dof list: entry (p, m) <- state entry (dofs[p], m)
  const std::vector<int32_t>& dofs = boundary_dofs(w->bnd);
  const int nv = w->nv;
  const size_t nbv = dofs.size() * (size_t)nv;
  std::vector<double> a(nbv, 1.0), d(nbv, 0.0);
  for (size_t p = 0; p < dofs.size(); ++p)
    for (int m = 0; m < nv; ++m)
    {
      const size_t i = (size_t)dofs[p] * nv + m;
      if (amp_host) a[p * nv + m] = amp_host[i];
      if (delay_host) d[p * nv + m] = delay_host[i];
    }
  // each buffer on its own: after a failed allocation (out of memory) a retry allocates what is missing
  if (w->prof_amp.n != nbv) w->prof_amp.alloc(nbv);
  if (w->prof_delay.n != nbv) w->prof_delay.alloc(nbv);
  w->prof_amp.upload(a);
  w->prof_delay.upload(d);
  w->prof_on = true;
  WFX_API_END
}

extern "C" int wfx_wave_set_snapshot(wfx_wave* w, int64_t every, wfx_snapshot_fn fn, void* user)
{
  WFX_API_BEGIN
  if (!w) fail("wave model is NULL");
  if (every < 0) fail("snapshot interval must not be negative");
  if (w->ens) fail("wave: snapshots are not available for ensemble models");
  ScopedDevice sd(w->ctx->device);
  flush_snapshot(w);
  w->snap_every = fn ? every : 0;
  w->snap_fn = fn;
  w->snap_user = user;
  if (w->snap_every > 0 && !w->snap_stream)
  {
    const size_t nb = (size_t)w->n * (w->dtype == WFX_F64 ? 8 : 4);
    w->snap_u.alloc(nb);
    w->snap_v.alloc(nb);
    WFX_CUDA(cudaMallocHost(&w->snap_hu, nb ? nb : 1));
    WFX_CUDA(cudaMallocHost(&w->snap_hv, nb ? nb : 1));
    WFX_CUDA(cudaStreamCreateWithFlags(&w->snap_stream, cudaStreamNonBlocking));
    WFX_CUDA(cudaEventCreateWithFlags(&w->ev_snap_ready, cudaEventDisableTiming));
    WFX_CUDA(cudaEventCreateWithFlags(&w->ev_snap_done, cudaEventDisableTiming));
  }
  WFX_API_END
}

extern "C" int wfx_wave_destroy(wfx_wave* w)
{
  WFX_API_BEGIN
  if (w)
  {
    ScopedDevice sd(w->ctx->device);
    delete w;
  }
  WFX_API_END
}
