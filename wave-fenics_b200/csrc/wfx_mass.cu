// Diagonal (GLL-collocated) mass operator, its inverse, and the atomic-free dofmap
// gather / scatter-add primitives.
//   wfx_mass_*         <- MassOperatorCPU (common/operators.hpp:43-109),
//                         SpectralMassOperator (common/cuda/spectral_mass.hpp:23-99)
//   wfx_gather         <- gather<T>  (common/cuda/scatter.cu:5-11,47-55)
//   wfx_scatter_add    <- scatter<T> (common/cuda/scatter.cu:38-45,57-65), atomics replaced
//                         by a segmented reduction over a precomputed inverse map
#include "wfx_internal.h"

#include <algorithm>
#include <cmath>

using namespace wfx;

namespace wfx
{
void build_tensor_dofmap(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap,
                         std::vector<int32_t>& tdm);
}

struct wfx_scatter_plan
{
  wfx_ctx* ctx = nullptr;
  int64_t n = 0, nout = 0;
  DevBuf<int64_t> d_off; // [nout+1]
  DevBuf<int32_t> d_src; // [n] source positions grouped by output entry, ascending
};

struct wfx_mass
{
  wfx_ctx* ctx = nullptr;
  int dtype = WFX_F64;
  int64_t ndofs = 0;
  DevBuf<double> d_m64; // always fp64
  void* d_m = nullptr;  // dtype T (aliases d_m64 for fp64)
  void* d_minv = nullptr;
  DevBuf<unsigned char> d_hx, d_hy;
  bool assembled = false; // diagonal summed over the ranks (wfx_mass_assemble)
  ~wfx_mass()
  {
    if (d_minv) cudaFree(d_minv);
    if (d_m && d_m != (void*)d_m64.p) cudaFree(d_m);
  }
};

namespace
{
template <typename T>
__global__ void gather_kernel(int64_t n, const int32_t* __restrict__ idx, const T* __restrict__ in,
                              T* __restrict__ out)
{
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[idx[i]];
}

// one thread per output entry; contributions added in ascending source position
template <typename TI, typename TO>
__global__ void segsum_kernel(int64_t nout, const int64_t* __restrict__ off,
                              const int32_t* __restrict__ src, const TI* __restrict__ in,
                              TO* __restrict__ out, int beta)
{
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= nout) return;
  TO s = beta ? out[j] : TO(0);
  for (int64_t p = off[j]; p < off[j + 1]; ++p) s += (TO)in[src[p]];
  out[j] = s;
}

// the weighted lumped mass (wfx_mass_create_weighted): segsum_kernel's reduction in the same order, every
// contribution in[p] scaled by its cell's weight w[p / nq] first.  __dmul_rn keeps nvcc from contracting the product
// into an FMA with the running sum, so that each term is rounded on its own as in a sum over w_c * detJw.
__global__ void segsum_weighted_kernel(int64_t nout, const int64_t* __restrict__ off, const int32_t* __restrict__ src,
                                       const double* __restrict__ in, const double* __restrict__ w, int nq,
                                       double* __restrict__ out)
{
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= nout) return;
  double s = 0.0;
  for (int64_t p = off[j]; p < off[j + 1]; ++p)
  {
    const int32_t q = src[p];
    s += __dmul_rn(w[q / nq], in[q]);
  }
  out[j] = s;
}

template <typename T>
__global__ void mass_finish_kernel(int64_t n, const double* __restrict__ m64, T* __restrict__ m,
                                   T* __restrict__ minv)
{
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double v = m64[i];
  if (m) m[i] = (T)v;
  minv[i] = v != 0.0 ? (T)(1.0 / v) : T(0);
}

template <typename T>
__global__ void diag_apply_kernel(int64_t n, const T* __restrict__ m, const T* __restrict__ x,
                                  T* __restrict__ y, int beta)
{
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const T v = m[i] * x[i];
  y[i] = beta ? y[i] + v : v;
}

void build_scatter_plan(wfx_scatter_plan* p, int64_t n, const int32_t* idx, int64_t nout)
{
  if (n >= (1ll << 31)) fail("scatter plan: more than 2^31 sources");
  std::vector<int64_t> off((size_t)nout + 1, 0);
  for (int64_t i = 0; i < n; ++i)
  {
    if (idx[i] < 0 || idx[i] >= nout) fail("scatter plan: index out of range");
    off[idx[i] + 1]++;
  }
  for (int64_t j = 0; j < nout; ++j) off[j + 1] += off[j];
  std::vector<int32_t> src((size_t)n);
  std::vector<int64_t> pos(off.begin(), off.end() - 1);
  for (int64_t i = 0; i < n; ++i) src[pos[idx[i]]++] = (int32_t)i; // ascending within a segment
  p->n = n;
  p->nout = nout;
  p->d_off.upload(off);
  p->d_src.upload(src);
}
} // namespace

extern "C" int wfx_gather(wfx_ctx* ctx, int dtype, int64_t n, const int32_t* idx, const void* in,
                          void* out, void* stream)
{
  WFX_API_BEGIN
  if (!ctx) fail("ctx is NULL");
  if (n <= 0) return 0;
  ScopedDevice sd(ctx->device);
  const unsigned grid = (unsigned)((n + 255) / 256);
  if (dtype == WFX_F64)
    gather_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(n, idx, (const double*)in, (double*)out);
  else if (dtype == WFX_F32)
    gather_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(n, idx, (const float*)in, (float*)out);
  else fail("unknown dtype %d", dtype);
  WFX_CUDA(cudaGetLastError());
  WFX_API_END
}

extern "C" int wfx_scatter_plan_create(wfx_ctx* ctx, int64_t n, const int32_t* idx_host,
                                       int64_t nout, wfx_scatter_plan** out)
{
  WFX_API_BEGIN
  if (!ctx || !out) fail("NULL argument");
  if (n < 0 || nout < 0) fail("negative size");
  ScopedDevice sd(ctx->device);
  auto p = std::make_unique<wfx_scatter_plan>();
  p->ctx = ctx;
  build_scatter_plan(p.get(), n, idx_host, nout);
  *out = p.release();
  WFX_API_END
}

extern "C" int wfx_scatter_add(wfx_scatter_plan* p, int dtype, const void* in, void* out, int beta,
                               void* stream)
{
  WFX_API_BEGIN
  if (!p) fail("scatter plan is NULL");
  if (p->nout == 0) return 0;
  ScopedDevice sd(p->ctx->device);
  const unsigned grid = (unsigned)((p->nout + 255) / 256);
  if (dtype == WFX_F64)
    segsum_kernel<double, double><<<grid, 256, 0, (cudaStream_t)stream>>>(
        p->nout, p->d_off.p, p->d_src.p, (const double*)in, (double*)out, beta);
  else if (dtype == WFX_F32)
    segsum_kernel<float, float><<<grid, 256, 0, (cudaStream_t)stream>>>(
        p->nout, p->d_off.p, p->d_src.p, (const float*)in, (float*)out, beta);
  else fail("unknown dtype %d", dtype);
  WFX_CUDA(cudaGetLastError());
  WFX_API_END
}

extern "C" int wfx_scatter_plan_destroy(wfx_scatter_plan* p)
{
  WFX_API_BEGIN
  if (p)
  {
    ScopedDevice sd(p->ctx->device);
    delete p;
  }
  WFX_API_END
}

extern "C" int wfx_mass_create(wfx_ctx* ctx, wfx_geom* geom, int64_t ndofs,
                               const int32_t* dofmap_host, wfx_mass** out)
{
  return wfx_mass_create_weighted(ctx, geom, ndofs, dofmap_host, nullptr, out);
}

extern "C" int wfx_mass_create_weighted(wfx_ctx* ctx, wfx_geom* geom, int64_t ndofs, const int32_t* dofmap_host,
                                        const double* cell_weight, wfx_mass** out)
{
  WFX_API_BEGIN
  if (!ctx || !geom || !out) fail("NULL argument");
  if (geom->ctx != ctx) fail("geometry belongs to another context");
  if (ndofs < 0) fail("negative ndofs");
  if (cell_weight)
    for (int64_t c = 0; c < geom->ncells; ++c)
      if (!std::isfinite(cell_weight[c]) || !(cell_weight[c] > 0))
        fail("weighted mass: the weight of cell %lld must be positive and finite", (long long)c);
  ScopedDevice sd(ctx->device);
  auto op = std::make_unique<wfx_mass>();
  op->ctx = ctx;
  op->dtype = geom->dtype;
  op->ndofs = ndofs;
  op->d_m64.alloc((size_t)ndofs);
  if (ndofs) WFX_CUDA(cudaMemset(op->d_m64.p, 0, (size_t)ndofs * 8));
  if (geom->ncells > 0 && ndofs > 0)
  {
    if (!dofmap_host) fail("dofmap is NULL");
    // m = M.1 (LinearGLL.hpp:102-110): m[dof(c,perm[t])] += detJ[c,t], cells in order.
    // The k-major tensor dofmap indexes dJw directly.
    SetupTimer timer("mass_create");
    std::vector<int32_t> tdm;
    build_tensor_dofmap(geom->P, geom->ncells, ndofs, dofmap_host, tdm);
    timer.lap("tensor dofmap");
    wfx_scatter_plan plan;
    plan.ctx = ctx;
    build_scatter_plan(&plan, (int64_t)tdm.size(), tdm.data(), ndofs);
    timer.lap("scatter plan");
    // m~ = sum_c w_c (detJ w)_{c,i}: the same segments, each contribution weighted by its cell (d_w lives until
    // the synchronisation below)
    DevBuf<double> d_w;
    if (cell_weight)
    {
      d_w.upload(cell_weight, (size_t)geom->ncells);
      segsum_weighted_kernel<<<(unsigned)((ndofs + 255) / 256), 256>>>(ndofs, plan.d_off.p, plan.d_src.p, geom->dJw,
                                                                       d_w.p, geom->nq, op->d_m64.p);
    }
    else
      segsum_kernel<double, double><<<(unsigned)((ndofs + 255) / 256), 256>>>(
          ndofs, plan.d_off.p, plan.d_src.p, geom->dJw, op->d_m64.p, 0);
    WFX_CUDA(cudaGetLastError());
    WFX_CUDA(cudaDeviceSynchronize());
  }
  const size_t esz = op->dtype == WFX_F64 ? 8 : 4;
  if (ndofs)
  {
    WFX_CUDA(cudaMalloc(&op->d_minv, (size_t)ndofs * esz));
    const unsigned grid = (unsigned)((ndofs + 255) / 256);
    if (op->dtype == WFX_F64)
    {
      op->d_m = op->d_m64.p;
      mass_finish_kernel<double><<<grid, 256>>>(ndofs, op->d_m64.p, nullptr, (double*)op->d_minv);
    }
    else
    {
      WFX_CUDA(cudaMalloc(&op->d_m, (size_t)ndofs * esz));
      mass_finish_kernel<float><<<grid, 256>>>(ndofs, op->d_m64.p, (float*)op->d_m, (float*)op->d_minv);
    }
    WFX_CUDA(cudaGetLastError());
    WFX_CUDA(cudaDeviceSynchronize());
  }
  *out = op.release();
  WFX_API_END
}

extern "C" int wfx_mass_apply(wfx_mass* op, const void* x, void* y, int beta, void* stream)
{
  WFX_API_BEGIN
  if (!op) fail("mass operator is NULL");
  if (op->ndofs == 0) return 0;
  if (!x || !y) fail("mass: NULL vector");
  ScopedDevice sd(op->ctx->device);
  const unsigned grid = (unsigned)((op->ndofs + 255) / 256);
  if (op->dtype == WFX_F64)
    diag_apply_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(
        op->ndofs, (const double*)op->d_m, (const double*)x, (double*)y, beta);
  else
    diag_apply_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(
        op->ndofs, (const float*)op->d_m, (const float*)x, (float*)y, beta);
  WFX_CUDA(cudaGetLastError());
  WFX_API_END
}

extern "C" int wfx_mass_apply_host(wfx_mass* op, const void* x_host, void* y_host, int beta)
{
  WFX_API_BEGIN
  if (!op) fail("mass operator is NULL");
  if (op->ndofs == 0) return 0;
  if (!x_host || !y_host) fail("mass: NULL vector");
  ScopedDevice sd(op->ctx->device);
  const size_t nb = (size_t)op->ndofs * (op->dtype == WFX_F64 ? 8 : 4);
  if (op->d_hx.n < nb) op->d_hx.alloc(nb);
  if (op->d_hy.n < nb) op->d_hy.alloc(nb);
  WFX_CUDA(cudaMemcpy(op->d_hx.p, x_host, nb, cudaMemcpyHostToDevice));
  if (beta) WFX_CUDA(cudaMemcpy(op->d_hy.p, y_host, nb, cudaMemcpyHostToDevice));
  if (wfx_mass_apply(op, op->d_hx.p, op->d_hy.p, beta, nullptr)) fail("%s", wfx_last_error());
  WFX_CUDA(cudaMemcpy(y_host, op->d_hy.p, nb, cudaMemcpyDeviceToHost));
  WFX_API_END
}

extern "C" int wfx_mass_apply_inverse(wfx_mass* op, const void* x, void* y, void* stream)
{
  WFX_API_BEGIN
  if (!op) fail("mass operator is NULL");
  if (op->ndofs == 0) return 0;
  if (!x || !y) fail("mass: NULL vector");
  ScopedDevice sd(op->ctx->device);
  const unsigned grid = (unsigned)((op->ndofs + 255) / 256);
  if (op->dtype == WFX_F64)
    diag_apply_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(
        op->ndofs, (const double*)op->d_minv, (const double*)x, (double*)y, 0);
  else
    diag_apply_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(
        op->ndofs, (const float*)op->d_minv, (const float*)x, (float*)y, 0);
  WFX_CUDA(cudaGetLastError());
  WFX_API_END
}

extern "C" int wfx_mass_assemble(wfx_mass* op, wfx_halo* halo)
{
  WFX_API_BEGIN
  if (!op || !halo) fail("NULL argument");
  // the diagonal is reduced in fp64 whatever the operator's dtype: an fp32 halo would
  // reinterpret the doubles (the model's own halo is not usable here for fp32 models)
  if (halo_dtype(halo) != WFX_F64) fail("mass assemble: needs an fp64 halo (the diagonal is summed in fp64)");
  if (op->assembled) return 0; // idempotent
  if (op->ndofs == 0)
  {
    op->assembled = true;
    return 0;
  }
  ScopedDevice sd(op->ctx->device);
  if (wfx_halo_update_rev_fwd(halo, op->d_m64.p, nullptr)) fail("%s", wfx_last_error());
  const unsigned grid = (unsigned)((op->ndofs + 255) / 256);
  if (op->dtype == WFX_F64)
    mass_finish_kernel<double><<<grid, 256>>>(op->ndofs, op->d_m64.p, nullptr, (double*)op->d_minv);
  else
    mass_finish_kernel<float><<<grid, 256>>>(op->ndofs, op->d_m64.p, (float*)op->d_m, (float*)op->d_minv);
  WFX_CUDA(cudaGetLastError());
  WFX_CUDA(cudaDeviceSynchronize());
  op->assembled = true; // only after the reduction succeeded: a failed call can be repeated
  WFX_API_END
}

namespace wfx
{
bool mass_assembled(const wfx_mass* op) { return op->assembled; }
int mass_dtype(const wfx_mass* op) { return op->dtype; }
int64_t mass_ndofs(const wfx_mass* op) { return op->ndofs; }
const double* mass_diagonal64(const wfx_mass* op) { return op->d_m64.p; }
} // namespace wfx

extern "C" int wfx_mass_diagonal(wfx_mass* op, const void** m)
{
  WFX_API_BEGIN
  if (!op || !m) fail("NULL argument");
  *m = op->d_m;
  WFX_API_END
}

extern "C" int wfx_mass_inverse_diagonal(wfx_mass* op, const void** minv)
{
  WFX_API_BEGIN
  if (!op || !minv) fail("NULL argument");
  *minv = op->d_minv;
  WFX_API_END
}

extern "C" int wfx_mass_destroy(wfx_mass* op)
{
  WFX_API_BEGIN
  if (op)
  {
    ScopedDevice sd(op->ctx->device);
    delete op;
  }
  WFX_API_END
}
