// Thermal model (DESIGN.md section 4.5d): the Pennes bioheat equation on the wave model's GLL mesh, classical
// RK4 on the device, and the CEM43 thermal dose.  The state is the rise theta = T - T_art.  A stage is one fused
// stiffness apply, b = scale .* (-cK^2 K theta_n) with scale = (k / cK^2) / (rhoC m), and one fused pointwise
// kernel that forms kv = b - r theta_n + f, both solution updates and the next stage state; stage 3 also adds the
// step's dose and the peak rise from the final theta held in registers.  Every other term is diagonal and folded
// into r and f at set-up.
#include "wfx_internal.h"

#include <cmath>
#include <cstdlib>

using namespace wfx;

struct wfx_thermal
{
  wfx_ctx* ctx = nullptr;
  wfx_stiffness* stiff = nullptr;
  wfx_mass* mass = nullptr;
  wfx_boundary* bnd = nullptr;
  int dtype = WFX_F64;
  int64_t n = 0;
  double T_art = 0, s = 1.0;
  const double* m64 = nullptr; // the mass operator's fp64 diagonal
  // th: solution; th0: start of step; thn: stage state; b: scaled stiffness result; scale, r, f: the diagonal
  // terms (model dtype)
  DevBuf<unsigned char> th, th0, thn, b, scale, r, f;
  // fp64: cap = rhoC m, fb = h1 m1 (T_ext1 - T_art) + h2 m2 (T_ext2 - T_art), q = Q; f = (fb + s q m) / cap
  DevBuf<double> cap, fb, q;
  // dose: CEM43 (fp64) and the peak rise (model dtype), reset by init / set_state
  DevBuf<double> cem;
  DevBuf<unsigned char> thmax;
  int64_t steps_done = 0;
  // power iteration: per-block partial sums and their totals
  DevBuf<double> red_part, red_sum;
  // one-rank graph replay of a whole step, captured per step size (the step reads no time: nothing is written
  // into the graph between replays)
  bool use_graph = true;
  cudaGraphExec_t step_graph = nullptr;
  double graph_dt = 0;
  cudaStream_t own_stream = nullptr;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  size_t esz() const { return dtype == WFX_F64 ? 8 : 4; }
  ~wfx_thermal()
  {
    if (step_graph) cudaGraphExecDestroy(step_graph);
    if (own_stream) cudaStreamDestroy(own_stream);
    if (ev_in) cudaEventDestroy(ev_in);
    if (ev_out) cudaEventDestroy(ev_out);
  }
};

namespace
{
constexpr int RED_BLOCKS = 592; // 4 per SM of a B200; a fixed grid keeps the reduction order fixed
// the RK4 stability interval on the negative real axis: |1 + z + z^2/2 + z^3/6 + z^4/24| <= 1 for z in [-x, 0]
constexpr double RK4_REAL_LIMIT = 2.785293563405282;

// Stage update (the tableau of rk_stage_kernel, wfx_wave.cu).  STAGE 0 reads the solution as stage state and
// saves it as th0; STAGE 3 finishes the solution and adds the step's dose:
//   kv = b - r thn + f,   th += b_i dt kv,   thn' = th0 + a_{i+1} dt kv
//   CEM43 += (dt / 60) R^(43 - T),  T = T_art + th,  R^(43 - T) = 2^(T - 43) (T >= 43) or 2^(2 (T - 43))
template <typename T, int STAGE>
__global__ void __launch_bounds__(256)
thermal_stage_kernel(int64_t n, const T* __restrict__ b, const T* __restrict__ r, const T* __restrict__ f,
                     T* __restrict__ th, T* __restrict__ th0, T* __restrict__ thn, T bdt, T adt_next, double dose_dt,
                     double T_art, double* __restrict__ cem, T* __restrict__ thmax)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n) return;
  const T ts = th[k];
  T x, base;
  if (STAGE == 0)
  {
    x = ts;
    base = ts;
    th0[k] = ts;
  }
  else
  {
    x = thn[k];
    if (STAGE < 3) base = th0[k];
  }
  const T kv = b[k] - r[k] * x + f[k];
  const T tn = kv * bdt + ts;
  th[k] = tn;
  if (STAGE < 3) thn[k] = kv * adt_next + base;
  else
  {
    const double e = (T_art + (double)tn) - 43.0;
    cem[k] += dose_dt * exp2(e >= 0.0 ? e : 2.0 * e);
    const T a = thmax[k];
    thmax[k] = (tn > a || tn != tn) ? tn : a; // NaN propagates, as in field_stats_kernel
  }
}

template <typename T>
void launch_stage(const wfx_thermal* th, int stage, double bdt, double adt_next, double dose_dt, cudaStream_t st)
{
  const unsigned grid = (unsigned)((th->n + 255) / 256);
#define WFX_STAGE(S)                                                                                                 \
  thermal_stage_kernel<T, S><<<grid, 256, 0, st>>>(th->n, (const T*)th->b.p, (const T*)th->r.p, (const T*)th->f.p,  \
                                                   (T*)th->th.p, (T*)th->th0.p, (T*)th->thn.p, (T)bdt, (T)adt_next, \
                                                   dose_dt, th->T_art, th->cem.p, (T*)th->thmax.p)
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

// out = out - r theta + f, out holding scale .* (-cK^2 K theta): the right-hand side on its own
template <typename T>
__global__ void thermal_rhs_kernel(int64_t n, const T* __restrict__ theta, const T* __restrict__ r,
                                   const T* __restrict__ f, T* __restrict__ out)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < n) out[k] = out[k] - r[k] * theta[k] + f[k];
}

// f = (fb + s Q m) / (rhoC m), whenever s or Q changes
template <typename T>
__global__ void thermal_source_kernel(int64_t n, const double* __restrict__ fb, const double* __restrict__ q,
                                      const double* __restrict__ m, const double* __restrict__ cap, double s,
                                      T* __restrict__ f)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < n) f[k] = (T)((fb[k] + s * q[k] * m[k]) / cap[k]);
}

// (h f0 / 1 MHz)^y / (rho0 c0) of harmonics h = 1..H, and the 2 / N of the amplitudes
struct HeatParams
{
  double c[WFX_HARMONICS_MAX];
  double amp_scale;
};
// Q_i = alpha0_i sum_h c_h |(2 / N) acc_h[i nv + m]|^2: one thread per dof, reading the H fp64 (re, im) planes of
// member m
__global__ void __launch_bounds__(256)
heat_source_kernel(int64_t n, int nv, int member, int nharm, const double2* __restrict__ harm, double alpha0,
                   const double* __restrict__ alpha0_dev, const __grid_constant__ HeatParams hp, double* __restrict__ q)
{
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t e = i * nv + member, plane = n * nv;
  double acc = 0.0;
#pragma unroll
  for (int h = 0; h < WFX_HARMONICS_MAX; ++h)
    if (h < nharm)
    {
      const double2 z = harm[h * plane + e];
      const double re = z.x * hp.amp_scale, im = z.y * hp.amp_scale;
      acc += hp.c[h] * (re * re + im * im);
    }
  q[i] = (alpha0_dev ? alpha0_dev[i] : alpha0) * acc;
}

template <typename T>
__global__ void fill_kernel(int64_t n, T v, T* __restrict__ x)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < n) x[k] = v;
}

// ---- power iteration ----------------------------------------------------------------------------------------
// start vector: a fixed hash of the index in [-1, 1)
template <typename T>
__global__ void pi_start_kernel(int64_t n, T* __restrict__ x)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n) return;
  uint64_t z = (uint64_t)k + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  x[k] = (T)((double)(z >> 11) * (2.0 / 9007199254740992.0) - 1.0);
}

// block sum of three fp64 values in a fixed tree order (blockDim.x == 256)
__device__ inline void block_sum3(double v0, double v1, double v2, double* out)
{
  __shared__ double sh[3][256];
  const int t = threadIdx.x;
  sh[0][t] = v0, sh[1][t] = v1, sh[2][t] = v2;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1)
  {
    if (t < w)
      for (int j = 0; j < 3; ++j) sh[j][t] += sh[j][t + w];
    __syncthreads();
  }
  if (t == 0) out[0] = sh[0][0], out[1] = sh[1][0], out[2] = sh[2][0];
}

// z = A x = r x - y, y = scale .* (-cK^2 K x) (written back into y), and the partial sums of the cap-weighted
// products x.z, x.x, z.z of this block's grid-stride entries
template <typename T>
__global__ void __launch_bounds__(256)
pi_apply_kernel(int64_t n, const T* __restrict__ x, T* __restrict__ y, const T* __restrict__ r,
                const double* __restrict__ cap, double* __restrict__ part)
{
  double s0 = 0, s1 = 0, s2 = 0;
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x)
  {
    const double xk = (double)x[k];
    const double z = (double)r[k] * xk - (double)y[k];
    const double w = cap[k];
    s0 += xk * w * z;
    s1 += xk * w * xk;
    s2 += z * w * z;
    y[k] = (T)z;
  }
  block_sum3(s0, s1, s2, part + 3 * blockIdx.x);
}

__global__ void __launch_bounds__(256) pi_total_kernel(int nblocks, const double* __restrict__ part, double* __restrict__ sum)
{
  double s0 = 0, s1 = 0, s2 = 0;
  for (int j = threadIdx.x; j < nblocks; j += blockDim.x)
    s0 += part[3 * j], s1 += part[3 * j + 1], s2 += part[3 * j + 2];
  block_sum3(s0, s1, s2, sum);
}

// x = z / |z|_cap
template <typename T>
__global__ void pi_normalise_kernel(int64_t n, const T* __restrict__ z, const double* __restrict__ sum, T* __restrict__ x)
{
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < n) x[k] = (T)((double)z[k] / sqrt(sum[2]));
}

// one step of size dt on st
void enqueue_step(wfx_thermal* th, double dt, cudaStream_t st)
{
  const double a_runge[5] = {0.0, 0.5, 0.5, 1.0, 0.0};
  const double b_runge[4] = {1.0 / 6.0, 1.0 / 3.0, 1.0 / 3.0, 1.0 / 6.0};
  static const char* const stage_name[4] = {"wfx thermal stage 0", "wfx thermal stage 1", "wfx thermal stage 2",
                                            "wfx thermal stage 3"};
  for (int i = 0; i < 4; ++i)
  {
    NvtxRange stage_range(stage_name[i]);
    const void* x = i == 0 ? th->th.p : th->thn.p;
    if (wfx_stiffness_apply_scaled(th->stiff, x, th->scale.p, th->b.p, st)) fail("%s", wfx_last_error());
    if (th->dtype == WFX_F64) launch_stage<double>(th, i, dt * b_runge[i], dt * a_runge[i + 1], dt / 60.0, st);
    else launch_stage<float>(th, i, dt * b_runge[i], dt * a_runge[i + 1], dt / 60.0, st);
  }
}

// f from fb, Q and s; ordered after and before all device work (steps may be in flight on any stream)
void update_source(wfx_thermal* th)
{
  WFX_CUDA(cudaDeviceSynchronize());
  if (th->n)
  {
    const unsigned grid = (unsigned)((th->n + 255) / 256);
    if (th->dtype == WFX_F64)
      thermal_source_kernel<double><<<grid, 256>>>(th->n, th->fb.p, th->q.p, th->m64, th->cap.p, th->s, (double*)th->f.p);
    else
      thermal_source_kernel<float><<<grid, 256>>>(th->n, th->fb.p, th->q.p, th->m64, th->cap.p, th->s, (float*)th->f.p);
    WFX_CUDA(cudaGetLastError());
  }
  WFX_CUDA(cudaDeviceSynchronize());
}

// CEM43 = 0, theta_max = -inf, no steps
void reset_dose(wfx_thermal* th)
{
  th->steps_done = 0;
  WFX_CUDA(cudaDeviceSynchronize());
  if (th->n)
  {
    WFX_CUDA(cudaMemsetAsync(th->cem.p, 0, th->n * sizeof(double), nullptr));
    const unsigned grid = (unsigned)((th->n + 255) / 256);
    if (th->dtype == WFX_F64) fill_kernel<double><<<grid, 256>>>(th->n, -INFINITY, (double*)th->thmax.p);
    else fill_kernel<float><<<grid, 256>>>(th->n, -INFINITY, (float*)th->thmax.p);
    WFX_CUDA(cudaGetLastError());
  }
  WFX_CUDA(cudaDeviceSynchronize());
}

void check_finite(const double* a, int64_t n, const char* what)
{
  for (int64_t i = 0; i < n; ++i)
    if (!std::isfinite(a[i])) fail("thermal: non-finite %s at entry %lld", what, (long long)i);
}
} // namespace

extern "C" int wfx_thermal_create(wfx_ctx* ctx, wfx_stiffness* stiff, wfx_mass* mass, wfx_boundary* bnd, double k,
                                  const double* rhoc, const double* perf, double T_art, const double* h_host,
                                  const double* T_ext_host, wfx_thermal** out)
{
  WFX_API_BEGIN
  if (!ctx || !stiff || !mass || !out || !rhoc) fail("NULL argument");
  ScopedDevice sd(ctx->device);
  int64_t ndofs = 0;
  if (wfx_stiffness_info(stiff, nullptr, nullptr, &ndofs, nullptr, nullptr, nullptr, nullptr))
    fail("%s", wfx_last_error());
  const int dtype = stiffness_dtype(stiff);
  if (mass_dtype(mass) != dtype) fail("thermal: mass operator dtype differs from the stiffness operator's");
  if (bnd && boundary_dtype(bnd) != dtype) fail("thermal: boundary operator dtype differs from the stiffness operator's");
  if (mass_ndofs(mass) != ndofs) fail("thermal: the mass operator has %lld dofs, the stiffness operator %lld",
                                      (long long)mass_ndofs(mass), (long long)ndofs);
  if (bnd && boundary_ndofs(bnd) != ndofs)
    fail("thermal: the boundary operator has %lld dofs, the stiffness operator %lld", (long long)boundary_ndofs(bnd),
         (long long)ndofs);
  if (stiffness_nshared(stiff) > 0) fail("thermal: one rank only (the stiffness operator has rank-shared dofs)");
  if (!std::isfinite(k) || !std::isfinite(T_art)) fail("thermal: non-finite k or T_art");
  if (!(k > 0)) fail("thermal: conductivity k must be positive");
  const double h[2] = {h_host ? h_host[0] : 0.0, h_host ? h_host[1] : 0.0};
  const double Te[2] = {T_ext_host ? T_ext_host[0] : T_art, T_ext_host ? T_ext_host[1] : T_art};
  check_finite(h, 2, "h");
  check_finite(Te, 2, "T_ext");
  if (h[0] < 0 || h[1] < 0) fail("thermal: heat transfer coefficients h must not be negative");
  if ((h[0] != 0 || h[1] != 0) && !bnd) fail("thermal: h != 0 needs a boundary operator");
  check_finite(rhoc, ndofs, "rhoC");
  for (int64_t i = 0; i < ndofs; ++i)
    if (!(rhoc[i] > 0)) fail("thermal: rhoC must be positive (entry %lld)", (long long)i);
  if (perf)
  {
    check_finite(perf, ndofs, "perfusion");
    for (int64_t i = 0; i < ndofs; ++i)
      if (perf[i] < 0) fail("thermal: perfusion must not be negative (entry %lld)", (long long)i);
  }
  auto th = std::make_unique<wfx_thermal>();
  th->ctx = ctx;
  th->stiff = stiff;
  th->mass = mass;
  th->bnd = bnd;
  th->dtype = dtype;
  th->n = ndofs;
  th->T_art = T_art;
  th->m64 = mass_diagonal64(mass);
  // the diagonal terms, in fp64 on the host
  const size_t n = (size_t)ndofs;
  std::vector<double> m(n), m1(n, 0.0), m2(n, 0.0);
  if (n) WFX_CUDA(cudaMemcpy(m.data(), th->m64, n * sizeof(double), cudaMemcpyDeviceToHost));
  if (bnd && wfx_boundary_get(bnd, m1.data(), m2.data())) fail("%s", wfx_last_error());
  const double cK = stiffness_c0(stiff), kk = k / (cK * cK);
  std::vector<double> cap(n), fb(n), scale(n), r(n);
  for (size_t i = 0; i < n; ++i)
  {
    cap[i] = rhoc[i] * m[i];
    scale[i] = kk / cap[i];
    r[i] = ((perf ? perf[i] : 0.0) * m[i] + h[0] * m1[i] + h[1] * m2[i]) / cap[i];
    fb[i] = h[0] * m1[i] * (Te[0] - T_art) + h[1] * m2[i] * (Te[1] - T_art);
  }
  const size_t nb = n * th->esz();
  for (auto* v : {&th->th, &th->th0, &th->thn, &th->b, &th->scale, &th->r, &th->f, &th->thmax})
  {
    v->alloc(nb);
    if (nb) WFX_CUDA(cudaMemset(v->p, 0, nb));
  }
  auto upload_t = [&](DevBuf<unsigned char>& dst, const std::vector<double>& src) {
    if (!n) return;
    if (dtype == WFX_F64) WFX_CUDA(cudaMemcpy(dst.p, src.data(), nb, cudaMemcpyHostToDevice));
    else
    {
      std::vector<float> tmp(src.begin(), src.end());
      WFX_CUDA(cudaMemcpy(dst.p, tmp.data(), nb, cudaMemcpyHostToDevice));
    }
  };
  upload_t(th->scale, scale);
  upload_t(th->r, r);
  th->cap.upload(cap);
  th->fb.upload(fb);
  th->q.alloc(n);
  th->cem.alloc(n);
  if (n) WFX_CUDA(cudaMemset(th->q.p, 0, n * sizeof(double)));
  th->red_part.alloc(3 * RED_BLOCKS);
  th->red_sum.alloc(3);
  if (const char* e = std::getenv("WFX_WAVE_GRAPH")) th->use_graph = std::atoi(e) != 0;
  WFX_CUDA(cudaStreamCreateWithFlags(&th->own_stream, cudaStreamNonBlocking));
  WFX_CUDA(cudaEventCreateWithFlags(&th->ev_in, cudaEventDisableTiming));
  WFX_CUDA(cudaEventCreateWithFlags(&th->ev_out, cudaEventDisableTiming));
  update_source(th.get());
  reset_dose(th.get());
  *out = th.release();
  WFX_API_END
}

extern "C" int wfx_thermal_init(wfx_thermal* th)
{
  WFX_API_BEGIN
  if (!th) fail("thermal model is NULL");
  ScopedDevice sd(th->ctx->device);
  WFX_CUDA(cudaDeviceSynchronize());
  if (th->th.n) WFX_CUDA(cudaMemset(th->th.p, 0, th->th.n));
  reset_dose(th);
  WFX_API_END
}

extern "C" int wfx_thermal_set_state(wfx_thermal* th, const void* theta)
{
  WFX_API_BEGIN
  if (!th) fail("thermal model is NULL");
  if (!theta) fail("thermal: NULL state");
  ScopedDevice sd(th->ctx->device);
  WFX_CUDA(cudaDeviceSynchronize());
  if (th->th.n) WFX_CUDA(cudaMemcpy(th->th.p, theta, th->th.n, cudaMemcpyHostToDevice));
  reset_dose(th);
  WFX_API_END
}

extern "C" int wfx_thermal_get_state(wfx_thermal* th, void* theta)
{
  WFX_API_BEGIN
  if (!th) fail("thermal model is NULL");
  if (!theta) fail("thermal: NULL state");
  ScopedDevice sd(th->ctx->device);
  WFX_CUDA(cudaDeviceSynchronize());
  if (th->th.n) WFX_CUDA(cudaMemcpy(theta, th->th.p, th->th.n, cudaMemcpyDeviceToHost));
  WFX_API_END
}

extern "C" int wfx_thermal_state_ptr(wfx_thermal* th, void** theta_dev)
{
  WFX_API_BEGIN
  if (!th || !theta_dev) fail("NULL argument");
  *theta_dev = th->th.p;
  WFX_API_END
}

extern "C" int wfx_thermal_set_heat_source(wfx_thermal* th, const double* q_host)
{
  WFX_API_BEGIN
  if (!th) fail("thermal model is NULL");
  if (q_host) check_finite(q_host, th->n, "heat source");
  ScopedDevice sd(th->ctx->device);
  WFX_CUDA(cudaDeviceSynchronize());
  if (th->n)
  {
    if (q_host) th->q.upload(q_host, (size_t)th->n);
    else WFX_CUDA(cudaMemset(th->q.p, 0, th->n * sizeof(double)));
  }
  update_source(th);
  WFX_API_END
}

extern "C" int wfx_thermal_heat_from_wave(wfx_thermal* th, wfx_wave* wave, int member, double alpha0,
                                          const double* alpha0_host, double y, double rho0, double c0)
{
  WFX_API_BEGIN
  if (!th || !wave) fail("NULL argument");
  const WaveFieldStats ws = wave_field_stats(wave);
  if (ws.ctx != th->ctx) fail("heat from wave: the wave model lives on another context");
  if (ws.ndofs != th->n) fail("heat from wave: the wave model has %lld dofs, the thermal model %lld",
                              (long long)ws.ndofs, (long long)th->n);
  if (!ws.on) fail("heat from wave: the wave model's field statistics are off (wfx_wave_set_field_stats)");
  if (ws.nharm == 0) fail("heat from wave: the field statistics keep no harmonics (nharm = 0)");
  if (ws.nsamples == 0) fail("heat from wave: the field statistics hold no samples yet (N = 0)");
  if (member < 0 || member >= ws.nv) fail("heat from wave: member %d outside [0, %d)", member, ws.nv);
  for (double x : {alpha0, y, rho0, c0})
    if (!std::isfinite(x)) fail("heat from wave: non-finite parameter");
  if (!(rho0 > 0) || !(c0 > 0)) fail("heat from wave: rho0 and c0 must be positive");
  if (alpha0 < 0) fail("heat from wave: alpha0 must not be negative");
  if (alpha0_host)
    for (int64_t i = 0; i < th->n; ++i)
      if (!std::isfinite(alpha0_host[i]) || alpha0_host[i] < 0)
        fail("heat from wave: alpha0 must be finite and not negative (entry %lld)", (long long)i);
  ScopedDevice sd(th->ctx->device);
  HeatParams hp{};
  for (int h = 1; h <= ws.nharm; ++h) hp.c[h - 1] = std::pow(h * ws.f0[member] / 1e6, y) / (rho0 * c0);
  hp.amp_scale = 2.0 / (double)ws.nsamples;
  DevBuf<double> a0;
  if (alpha0_host) a0.upload(alpha0_host, (size_t)th->n);
  WFX_CUDA(cudaDeviceSynchronize()); // the wave's steps and this model's steps may be in flight
  if (th->n)
  {
    const unsigned grid = (unsigned)((th->n + 255) / 256);
    heat_source_kernel<<<grid, 256>>>(th->n, ws.nv, member, ws.nharm, ws.harm, alpha0, a0.p, hp, th->q.p);
    WFX_CUDA(cudaGetLastError());
  }
  update_source(th);
  WFX_API_END
}

extern "C" int wfx_thermal_get_heat_source(wfx_thermal* th, double* q_host)
{
  WFX_API_BEGIN
  if (!th || !q_host) fail("NULL argument");
  ScopedDevice sd(th->ctx->device);
  WFX_CUDA(cudaDeviceSynchronize());
  th->q.download(q_host, (size_t)th->n);
  WFX_API_END
}

extern "C" int wfx_thermal_set_heat_scale(wfx_thermal* th, double s)
{
  WFX_API_BEGIN
  if (!th) fail("thermal model is NULL");
  if (!std::isfinite(s) || s < 0) fail("thermal: the heat scale s must be finite and not negative");
  ScopedDevice sd(th->ctx->device);
  th->s = s;
  update_source(th);
  WFX_API_END
}

extern "C" int wfx_thermal_rhs(wfx_thermal* th, const void* theta, void* out, void* stream)
{
  WFX_API_BEGIN
  if (!th) fail("thermal model is NULL");
  if (!theta || !out) fail("thermal rhs: NULL vector");
  if (theta == out) fail("thermal rhs: out must not alias theta");
  ScopedDevice sd(th->ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (wfx_stiffness_apply_scaled(th->stiff, theta, th->scale.p, out, st)) fail("%s", wfx_last_error());
  if (th->n == 0) return 0;
  const unsigned grid = (unsigned)((th->n + 255) / 256);
  if (th->dtype == WFX_F64)
    thermal_rhs_kernel<double><<<grid, 256, 0, st>>>(th->n, (const double*)theta, (const double*)th->r.p,
                                                     (const double*)th->f.p, (double*)out);
  else
    thermal_rhs_kernel<float><<<grid, 256, 0, st>>>(th->n, (const float*)theta, (const float*)th->r.p,
                                                    (const float*)th->f.p, (float*)out);
  WFX_CUDA(cudaGetLastError());
  WFX_API_END
}

extern "C" int wfx_thermal_rk4(wfx_thermal* th, double t0, double tf, double dt, int64_t max_steps, int64_t* steps_out,
                               double* t_end, void* stream)
{
  WFX_API_BEGIN
  if (!th) fail("thermal model is NULL");
  if (!std::isfinite(t0) || !std::isfinite(tf) || !std::isfinite(dt)) fail("thermal rk4: non-finite time");
  if (!(dt > 0)) fail("thermal rk4: dt must be positive");
  ScopedDevice sd(th->ctx->device);
  cudaStream_t st = (cudaStream_t)stream;
  // graph capture cannot use the legacy default stream: such callers are moved to the own stream, ordered by events
  const bool graph_ok = th->use_graph && stiffness_graph_safe(th->stiff);
  cudaStream_t ws = st;
  if (graph_ok && (st == nullptr || st == cudaStreamLegacy))
  {
    ws = th->own_stream;
    WFX_CUDA(cudaEventRecord(th->ev_in, st));
    WFX_CUDA(cudaStreamWaitEvent(ws, th->ev_in, 0));
  }
  double t = t0;
  int64_t step = 0;
  const double dt_nominal = dt;
  while (t < tf)
  {
    if (max_steps > 0 && step >= max_steps) break;
    NvtxRange step_range("wfx thermal step");
    dt = std::min(dt, tf - t);
    if (graph_ok && dt == dt_nominal && th->n)
    {
      if (!th->step_graph || th->graph_dt != dt)
      {
        if (th->step_graph) WFX_CUDA(cudaGraphExecDestroy(th->step_graph));
        th->step_graph = nullptr;
        cudaGraph_t graph = nullptr;
        WFX_CUDA(cudaStreamBeginCapture(ws, cudaStreamCaptureModeThreadLocal));
        try
        {
          enqueue_step(th, dt, ws);
        }
        catch (...)
        {
          cudaStreamEndCapture(ws, &graph);
          if (graph) cudaGraphDestroy(graph);
          throw;
        }
        WFX_CUDA(cudaStreamEndCapture(ws, &graph));
        const cudaError_t ie = cudaGraphInstantiate(&th->step_graph, graph, 0);
        cudaGraphDestroy(graph);
        WFX_CUDA(ie);
        th->graph_dt = dt;
      }
      WFX_CUDA(cudaGraphLaunch(th->step_graph, ws));
    }
    else if (th->n) enqueue_step(th, dt, ws);
    t += dt;
    step += 1;
    th->steps_done += 1;
  }
  if (ws != st)
  {
    WFX_CUDA(cudaEventRecord(th->ev_out, ws));
    WFX_CUDA(cudaStreamWaitEvent(st, th->ev_out, 0));
  }
  if (steps_out) *steps_out = step;
  if (t_end) *t_end = t;
  WFX_API_END
}

extern "C" int wfx_thermal_get_dose(wfx_thermal* th, int64_t* nsteps, double* cem43_host, void* theta_max_host)
{
  WFX_API_BEGIN
  if (!th) fail("thermal model is NULL");
  ScopedDevice sd(th->ctx->device);
  if (nsteps) *nsteps = th->steps_done;
  if (!cem43_host && !theta_max_host) return 0;
  WFX_CUDA(cudaDeviceSynchronize());
  if (cem43_host) th->cem.download(cem43_host, (size_t)th->n);
  if (theta_max_host && th->thmax.n) WFX_CUDA(cudaMemcpy(theta_max_host, th->thmax.p, th->thmax.n, cudaMemcpyDeviceToHost));
  WFX_API_END
}

extern "C" int wfx_thermal_stable_dt(wfx_thermal* th, int iters, double* lambda, double* dt_max)
{
  WFX_API_BEGIN
  if (!th) fail("thermal model is NULL");
  if (iters < 1) fail("thermal stable_dt: iters must be at least 1");
  ScopedDevice sd(th->ctx->device);
  if (th->n == 0) fail("thermal stable_dt: the model has no dofs");
  // thn and b are scratch between steps: x lives in thn, y = z in b
  WFX_CUDA(cudaDeviceSynchronize());
  const unsigned grid = (unsigned)((th->n + 255) / 256);
  const int nred = (int)std::min<int64_t>(RED_BLOCKS, (th->n + 255) / 256);
  for (int it = 0; it < iters; ++it)
  {
    if (th->dtype == WFX_F64)
    {
      if (it == 0) pi_start_kernel<double><<<grid, 256>>>(th->n, (double*)th->thn.p);
      else pi_normalise_kernel<double><<<grid, 256>>>(th->n, (const double*)th->b.p, th->red_sum.p, (double*)th->thn.p);
    }
    else
    {
      if (it == 0) pi_start_kernel<float><<<grid, 256>>>(th->n, (float*)th->thn.p);
      else pi_normalise_kernel<float><<<grid, 256>>>(th->n, (const float*)th->b.p, th->red_sum.p, (float*)th->thn.p);
    }
    WFX_CUDA(cudaGetLastError());
    if (wfx_stiffness_apply_scaled(th->stiff, th->thn.p, th->scale.p, th->b.p, nullptr)) fail("%s", wfx_last_error());
    if (th->dtype == WFX_F64)
      pi_apply_kernel<double><<<nred, 256>>>(th->n, (const double*)th->thn.p, (double*)th->b.p, (const double*)th->r.p,
                                             th->cap.p, th->red_part.p);
    else
      pi_apply_kernel<float><<<nred, 256>>>(th->n, (const float*)th->thn.p, (float*)th->b.p, (const float*)th->r.p,
                                            th->cap.p, th->red_part.p);
    pi_total_kernel<<<1, 256>>>(nred, th->red_part.p, th->red_sum.p);
    WFX_CUDA(cudaGetLastError());
  }
  double sums[3];
  WFX_CUDA(cudaMemcpy(sums, th->red_sum.p, sizeof(sums), cudaMemcpyDeviceToHost));
  const double lam = sums[0] / sums[1];
  if (!(lam > 0) || !std::isfinite(lam)) fail("thermal stable_dt: the power iteration gave lambda = %g", lam);
  if (lambda) *lambda = lam;
  if (dt_max) *dt_max = RK4_REAL_LIMIT / lam;
  WFX_API_END
}

extern "C" int wfx_thermal_destroy(wfx_thermal* th)
{
  WFX_API_BEGIN
  if (th)
  {
    ScopedDevice sd(th->ctx->device);
    cudaDeviceSynchronize();
    delete th;
  }
  WFX_API_END
}
