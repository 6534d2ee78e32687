// Boundary linear form of the wave model:  b += c0^2 g m1 - c0 m2 .* v_n
// (demo/cpu_planar3d/forms.ufl:21-24, assembled by fem::assemble_vector at
// common/LinearGLL.hpp:175).  With the GLL facet rule the form is diagonal; the facet
// masses m1 (tag 1, Neumann source) and m2 (tag 2, absorbing) are reduced once on the host
// over the tagged facets and kept compact (boundary dofs only) on the device.
#include "wfx_internal.h"
#include "wfx_source.h"

#include <cmath>
#include <map>

using namespace wfx;

struct wfx_boundary
{
  wfx_ctx* ctx = nullptr;
  int dtype = WFX_F64;
  int64_t ndofs = 0, nb = 0;
  DevBuf<int32_t> d_idx;
  DevBuf<double> d_m1, d_m2; // compact, fp64 (tiny)
  std::vector<int32_t> h_idx;
  std::vector<double> h_m1, h_m2;
  bool assembled = false; // facet masses summed over the ranks (wfx_boundary_assemble)
};

namespace
{
// g_dev (nullable): the source amplitude g in device memory; then c02g holds c0^2 and the product
// c0^2 * g is formed here with the same single rounding as on the host.
template <typename T>
__global__ void boundary_kernel(int64_t nb, const int32_t* __restrict__ idx,
                                const double* __restrict__ m1, const double* __restrict__ m2,
                                double c02g, double c0, const T* __restrict__ vn, T* __restrict__ b,
                                const double* __restrict__ g_dev)
{
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= nb) return;
  if (g_dev) c02g = __dmul_rn(c02g, *g_dev);
  const int32_t i = idx[t];
  b[i] = (T)((double)b[i] + c02g * m1[t] - c0 * m2[t] * (double)vn[i]);
}

// the same for nv member-interleaved fields, one thread per (boundary dof, member); c02 = c0^2 and the
// product c0^2 * g_m is rounded once as in boundary_kernel
struct EnsAmp
{
  double g[WFX_ENSEMBLE_MAX];
};
template <typename T>
__global__ void boundary_ens_kernel(int64_t nb, int nv, const int32_t* __restrict__ idx,
                                    const double* __restrict__ m1, const double* __restrict__ m2, double c02,
                                    double c0, const EnsAmp gh, const double* __restrict__ g_dev,
                                    const T* __restrict__ vn, T* __restrict__ b)
{
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= nb * nv) return;
  const int64_t p = t / nv;
  const int m = (int)(t % nv);
  const double c02g = __dmul_rn(c02, g_dev ? g_dev[m] : gh.g[m]);
  const int64_t i = (int64_t)idx[p] * nv + m;
  b[i] = (T)((double)b[i] + c02g * m1[p] - c0 * m2[p] * (double)vn[i]);
}

// A source profile (section 4.5c) on nv member-interleaved fields (nv = 1: one field), one thread per
// (boundary dof p, member m), compact entry t = p nv + m:
//   b[i,m] += c0^2 a_t (g_m + s_src g_m')(tn - tau_t) m1_p - c0 m2_p vn[i,m],   g_m = g_m' = 0 before tau_t,
// with g_m member m's source (f0, p0 of SourceParams) evaluated in fp64 by source_eval for every scalar type.
// The stage time tn comes by value or, in graph replays, from t_dev.  Entries off Gamma1 (m1 = 0) and
// switched-off entries (a = 0) skip the trigonometry.
template <typename T>
__global__ void __launch_bounds__(256)
boundary_profile_kernel(int64_t nb, int nv, const int32_t* __restrict__ idx, const double* __restrict__ m1,
                        const double* __restrict__ m2, double c0, double s_src, const __grid_constant__ SourceParams sp,
                        double t_host, const double* __restrict__ t_dev, const double* __restrict__ amp,
                        const double* __restrict__ delay, const T* __restrict__ vn, T* __restrict__ b)
{
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= nb * nv) return;
  const int64_t p = t / nv;
  const int m = (int)(t % nv);
  const double m1p = m1[p], a = amp[t];
  double src = 0.0;
  if (m1p != 0.0 && a != 0.0)
  {
    const double s = (t_dev ? *t_dev : t_host) - delay[t];
    if (s >= 0.0)
    {
      double g, gdot;
      source_eval(sp.f0[m], sp.p0[m], c0, s, &g, &gdot);
      src = a * (g + s_src * gdot);
    }
  }
  const int64_t i = (int64_t)idx[p] * nv + m;
  b[i] = (T)((double)b[i] + __dmul_rn(c0 * c0, src) * m1p - c0 * m2[p] * (double)vn[i]);
}

// Lossy / Westervelt models: the Gamma2 mass term q = qc m2 on the absorbing dofs only, so that the dense
// stage update needs nothing beyond 1/m (see boundary_absorbing_mass in wfx_internal.h).  p is formed in T
// exactly as the stage kernel forms it.
template <typename T>
__global__ void absorbing_mass_kernel(int64_t nb, const int32_t* __restrict__ idx, const double* __restrict__ m2,
                                      const double* __restrict__ m, double qc, double kappa, T s,
                                      const T* __restrict__ pw, const T* __restrict__ pd, T* __restrict__ b)
{
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= nb || m2[t] == 0.0) return;
  const int32_t i = idx[t];
  const T pdt = pd[i];
  const double p = (double)(pw[i] - s * pdt);
  const double mi = m[i], a = 1.0 - kappa * p, kp2 = kappa * (double)pdt * (double)pdt;
  const double kv = ((double)b[i] + mi * kp2) / (mi * a + qc * m2[t]);
  b[i] = (T)(mi * (kv * a - kp2));
}
} // namespace

void wfx::boundary_absorbing_mass(wfx_boundary* op, const double* m64, double qc, double kappa, double s,
                                  const void* pw, const void* pd, void* b, cudaStream_t stream)
{
  if (!op || op->nb == 0) return;
  const unsigned grid = (unsigned)((op->nb + 255) / 256);
  if (op->dtype == WFX_F64)
    absorbing_mass_kernel<double><<<grid, 256, 0, stream>>>(op->nb, op->d_idx.p, op->d_m2.p, m64, qc, kappa, s,
                                                             (const double*)pw, (const double*)pd, (double*)b);
  else
    absorbing_mass_kernel<float><<<grid, 256, 0, stream>>>(op->nb, op->d_idx.p, op->d_m2.p, m64, qc, kappa, (float)s,
                                                            (const float*)pw, (const float*)pd, (float*)b);
  WFX_CUDA(cudaGetLastError());
}

void wfx::boundary_apply_profile(wfx_boundary* op, int nv, double c0, double s_src, const SourceParams& sp,
                                 double t_host, const double* t_dev, const double* amp, const double* delay,
                                 const void* vn, void* b, cudaStream_t stream)
{
  if (!op || op->nb == 0) return;
  if (nv < 1 || nv > WFX_ENSEMBLE_MAX) fail("boundary: nv = %d outside [1, %d]", nv, WFX_ENSEMBLE_MAX);
  const unsigned grid = (unsigned)((op->nb * nv + 255) / 256);
  if (op->dtype == WFX_F64)
    boundary_profile_kernel<double><<<grid, 256, 0, stream>>>(op->nb, nv, op->d_idx.p, op->d_m1.p, op->d_m2.p, c0,
                                                               s_src, sp, t_host, t_dev, amp, delay,
                                                               (const double*)vn, (double*)b);
  else
    boundary_profile_kernel<float><<<grid, 256, 0, stream>>>(op->nb, nv, op->d_idx.p, op->d_m1.p, op->d_m2.p, c0,
                                                              s_src, sp, t_host, t_dev, amp, delay,
                                                              (const float*)vn, (float*)b);
  WFX_CUDA(cudaGetLastError());
}

void wfx::boundary_apply_ens(wfx_boundary* op, int nv, double c0, const double* g_host, const double* g_dev,
                             const void* vn, void* b, cudaStream_t stream)
{
  if (!op || op->nb == 0) return;
  if (nv < 1 || nv > WFX_ENSEMBLE_MAX) fail("boundary: nv = %d outside [1, %d]", nv, WFX_ENSEMBLE_MAX);
  EnsAmp gh{};
  if (!g_dev)
    for (int m = 0; m < nv; ++m) gh.g[m] = g_host[m];
  const unsigned grid = (unsigned)((op->nb * nv + 255) / 256);
  if (op->dtype == WFX_F64)
    boundary_ens_kernel<double><<<grid, 256, 0, stream>>>(op->nb, nv, op->d_idx.p, op->d_m1.p, op->d_m2.p, c0 * c0,
                                                           c0, gh, g_dev, (const double*)vn, (double*)b);
  else
    boundary_ens_kernel<float><<<grid, 256, 0, stream>>>(op->nb, nv, op->d_idx.p, op->d_m1.p, op->d_m2.p, c0 * c0,
                                                          c0, gh, g_dev, (const float*)vn, (float*)b);
  WFX_CUDA(cudaGetLastError());
}

extern "C" int wfx_boundary_create(wfx_ctx* ctx, int P, int dtype, int64_t nfacets,
                                   const int32_t* fcell, const int32_t* flocal,
                                   const int32_t* ftag, int64_t npts, const double* x,
                                   const int32_t* xdofs, int64_t ndofs, const int32_t* dofmap,
                                   wfx_boundary** out)
{
  WFX_API_BEGIN
  if (!ctx || !out) fail("NULL argument");
  if (P < 1 || P + 1 > WFX_MAXN) fail("degree %d out of range", P);
  if (dtype != WFX_F64 && dtype != WFX_F32) fail("unknown dtype %d", dtype);
  ScopedDevice sd(ctx->device);
  const int n = P + 1, nd = n * n * n;
  double pts[WFX_MAXN], wts[WFX_MAXN];
  gll_points_weights(P, pts, wts);
  std::vector<int32_t> perm(nd);
  tensor_perm(P, perm.data());
  // local facet -> (normal axis, side): DOLFINx hexahedron facets (0,1,2,3) z=0, (0,1,4,5) y=0,
  // (0,2,4,6) x=0, (1,3,5,7) x=1, (2,3,6,7) y=1, (4,5,6,7) z=1
  static const int NORMAL[6] = {2, 1, 0, 0, 1, 2}, SIDE[6] = {0, 0, 0, 1, 1, 1};
  std::map<int32_t, std::pair<double, double>> acc; // dof -> (m1, m2), facet order
  for (int64_t f = 0; f < nfacets; ++f)
  {
    const int tag = ftag[f];
    if (tag != 1 && tag != 2) continue;
    const int lf = flocal[f];
    if (lf < 0 || lf > 5) fail("local facet index %d out of range", lf);
    const int64_t c = fcell[f];
    const int na = NORMAL[lf], ta = na == 0 ? 1 : 0, tb = na == 2 ? 1 : 2;
    double xv[8][3];
    for (int v = 0; v < 8; ++v)
    {
      const int64_t g = xdofs[8 * c + v];
      if (g < 0 || g >= npts) fail("geometry dofmap entry out of range");
      for (int a = 0; a < 3; ++a) xv[v][a] = x[3 * g + a];
    }
    for (int ia = 0; ia < n; ++ia)
      for (int ib = 0; ib < n; ++ib)
      {
        int id[3];
        id[na] = SIDE[lf];
        id[ta] = ia;
        id[tb] = ib;
        const double X[3] = {pts[id[0]], pts[id[1]], pts[id[2]]};
        // tangent vectors d x / d X_ta, d x / d X_tb of the trilinear map
        double t1[3] = {0, 0, 0}, t2[3] = {0, 0, 0};
        for (int v = 0; v < 8; ++v)
        {
          double fac[3], sgn[3];
          for (int a = 0; a < 3; ++a)
          {
            const int bit = (v >> a) & 1;
            fac[a] = bit ? X[a] : 1.0 - X[a];
            sgn[a] = bit ? 1.0 : -1.0;
          }
          const double da = clamp_m101(sgn[ta] * fac[(ta + 1) % 3] * fac[(ta + 2) % 3]);
          const double db = clamp_m101(sgn[tb] * fac[(tb + 1) % 3] * fac[(tb + 2) % 3]);
          for (int a = 0; a < 3; ++a)
          {
            t1[a] += xv[v][a] * da;
            t2[a] += xv[v][a] * db;
          }
        }
        const double cx = t1[1] * t2[2] - t1[2] * t2[1];
        const double cy = t1[2] * t2[0] - t1[0] * t2[2];
        const double cz = t1[0] * t2[1] - t1[1] * t2[0];
        const double ds = wts[ia] * wts[ib] * std::sqrt(cx * cx + cy * cy + cz * cz);
        const int32_t dof = dofmap[c * nd + perm[(id[0] * n + id[1]) * n + id[2]]];
        if (dof < 0 || dof >= ndofs) fail("dofmap entry out of range");
        auto& e = acc[dof];
        (tag == 1 ? e.first : e.second) += ds;
      }
  }
  auto op = std::make_unique<wfx_boundary>();
  op->ctx = ctx;
  op->dtype = dtype;
  op->ndofs = ndofs;
  for (auto& kv : acc)
  {
    op->h_idx.push_back(kv.first);
    op->h_m1.push_back(kv.second.first);
    op->h_m2.push_back(kv.second.second);
  }
  op->nb = (int64_t)op->h_idx.size();
  if (op->nb)
  {
    op->d_idx.upload(op->h_idx);
    op->d_m1.upload(op->h_m1);
    op->d_m2.upload(op->h_m2);
  }
  *out = op.release();
  WFX_API_END
}

extern "C" int wfx_boundary_apply(wfx_boundary* op, double c0, double g, const void* vn, void* b,
                                  void* stream)
{
  WFX_API_BEGIN
  if (!op) fail("boundary operator is NULL");
  if (op->nb == 0) return 0;
  if (!vn || !b) fail("boundary: NULL vector");
  ScopedDevice sd(op->ctx->device);
  const unsigned grid = (unsigned)((op->nb + 255) / 256);
  const double c02g = c0 * c0 * g;
  if (op->dtype == WFX_F64)
    boundary_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(
        op->nb, op->d_idx.p, op->d_m1.p, op->d_m2.p, c02g, c0, (const double*)vn, (double*)b, nullptr);
  else
    boundary_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(
        op->nb, op->d_idx.p, op->d_m1.p, op->d_m2.p, c02g, c0, (const float*)vn, (float*)b, nullptr);
  WFX_CUDA(cudaGetLastError());
  WFX_API_END
}

void wfx::boundary_apply_dev(wfx_boundary* op, double c0, const double* g_dev, const void* vn, void* b,
                             cudaStream_t stream)
{
  if (!op || op->nb == 0) return;
  const unsigned grid = (unsigned)((op->nb + 255) / 256);
  const double c02 = c0 * c0;
  if (op->dtype == WFX_F64)
    boundary_kernel<double><<<grid, 256, 0, stream>>>(op->nb, op->d_idx.p, op->d_m1.p, op->d_m2.p, c02, c0,
                                                       (const double*)vn, (double*)b, g_dev);
  else
    boundary_kernel<float><<<grid, 256, 0, stream>>>(op->nb, op->d_idx.p, op->d_m1.p, op->d_m2.p, c02, c0,
                                                      (const float*)vn, (float*)b, g_dev);
  WFX_CUDA(cudaGetLastError());
}

extern "C" int wfx_boundary_get(wfx_boundary* op, double* m1, double* m2)
{
  WFX_API_BEGIN
  if (!op) fail("boundary operator is NULL");
  for (int64_t i = 0; i < op->ndofs; ++i)
  {
    if (m1) m1[i] = 0;
    if (m2) m2[i] = 0;
  }
  for (int64_t t = 0; t < op->nb; ++t)
  {
    if (m1) m1[op->h_idx[t]] = op->h_m1[t];
    if (m2) m2[op->h_idx[t]] = op->h_m2[t];
  }
  WFX_API_END
}

extern "C" int wfx_boundary_assemble(wfx_boundary* op, wfx_halo* halo)
{
  WFX_API_BEGIN
  if (!op || !halo) fail("NULL argument");
  if (halo_dtype(halo) != WFX_F64) fail("boundary assemble: needs an fp64 halo (facet masses are summed in fp64)");
  if (op->assembled) return 0; // idempotent
  ScopedDevice sd(op->ctx->device);
  // dense fp64 vectors through the ghost reduction, then compact again: a dof may carry a
  // boundary term here only because a neighbouring rank owns the tagged facet
  std::vector<double> m1((size_t)op->ndofs, 0.0), m2((size_t)op->ndofs, 0.0);
  for (int64_t t = 0; t < op->nb; ++t)
  {
    m1[op->h_idx[t]] = op->h_m1[t];
    m2[op->h_idx[t]] = op->h_m2[t];
  }
  DevBuf<double> d1((size_t)op->ndofs), d2((size_t)op->ndofs);
  d1.upload(m1);
  d2.upload(m2);
  if (op->ndofs)
  {
    if (wfx_halo_update_rev_fwd(halo, d1.p, nullptr)) fail("%s", wfx_last_error());
    if (wfx_halo_update_rev_fwd(halo, d2.p, nullptr)) fail("%s", wfx_last_error());
    WFX_CUDA(cudaDeviceSynchronize());
    d1.download(m1.data(), m1.size());
    d2.download(m2.data(), m2.size());
  }
  op->h_idx.clear();
  op->h_m1.clear();
  op->h_m2.clear();
  for (int64_t i = 0; i < op->ndofs; ++i)
    if (m1[i] != 0.0 || m2[i] != 0.0)
    {
      op->h_idx.push_back((int32_t)i);
      op->h_m1.push_back(m1[i]);
      op->h_m2.push_back(m2[i]);
    }
  op->nb = (int64_t)op->h_idx.size();
  if (op->nb)
  {
    op->d_idx.upload(op->h_idx);
    op->d_m1.upload(op->h_m1);
    op->d_m2.upload(op->h_m2);
  }
  op->assembled = true; // only after the reduction succeeded
  WFX_API_END
}

namespace wfx
{
bool boundary_assembled(const wfx_boundary* op) { return op->assembled; }
int boundary_dtype(const wfx_boundary* op) { return op->dtype; }
int64_t boundary_ndofs(const wfx_boundary* op) { return op->ndofs; }
const std::vector<int32_t>& boundary_dofs(const wfx_boundary* op) { return op->h_idx; }
} // namespace wfx

extern "C" int wfx_boundary_destroy(wfx_boundary* op)
{
  WFX_API_BEGIN
  if (op)
  {
    ScopedDevice sd(op->ctx->device);
    delete op;
  }
  WFX_API_END
}
