// Per-cell geometric-factor precompute on the GPU.
//   wfx_geometry_create      <- precompute_geometric_data (common/precomputation.hpp:18-110)
//   wfx_compute_jacobian_data <- compute_jacobian / _determinant / _inverse /
//                                compute_geometrical_factor (common/precompute.hpp:49-176)
// One thread per (cell, point).  All arithmetic is fp64 with explicit rounding
// (__dmul_rn/__dadd_rn/fma) in the reference's operation order, so the result does not
// depend on compiler contraction; G is stored symmetric (6 entries) in the layout the
// stiffness kernel streams.
#include "wfx_internal.h"
#include "wfx_plan.h"

#include <cmath>
#include <utility>

using namespace wfx;

wfx_geom::~wfx_geom()
{
  if (G6) cudaFree(G6);
  if (dJw) cudaFree(dJw);
  if (Gc) cudaFree(Gc);
  if (affine) cudaFree(affine);
}

namespace
{
struct Tables1D
{
  double pts[WFX_MAXN];
  double wts[WFX_MAXN];
};

__device__ __forceinline__ double clamp_dev(double v)
{
  // xt::isclose(v, t), rtol 1e-5, atol 1e-8, t = -1, 0, 1 in the reference's order
  if (fabs(v - (-1.0)) <= 1e-8 + 1e-5 * 1.0) v = -1.0;
  if (fabs(v - 0.0) <= 1e-8) v = 0.0;
  if (fabs(v - 1.0) <= 1e-8 + 1e-5 * 1.0) v = 1.0;
  return v;
}

// Kahan's difference of products a*d - b*c, as dolfinx::math does for det/inv.
__device__ __forceinline__ double diffprod(double a, double b, double c, double d)
{
  double w = __dmul_rn(b, c);
  double err = fma(-b, c, w);
  double diff = fma(a, d, -w);
  return __dadd_rn(diff, err);
}

// J[i][j] = sum_v coords[v][i] * dphi_j(v) for the trilinear hexahedron map at X.
template <bool CLAMP>
__device__ __forceinline__ void jacobian_at(const double* __restrict__ x,
                                            const int32_t* __restrict__ xd, const double X[3],
                                            double J[3][3])
{
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) J[i][j] = 0.0;
#pragma unroll
  for (int v = 0; v < 8; ++v)
  {
    double f[3], s[3], d[3];
#pragma unroll
    for (int a = 0; a < 3; ++a)
    {
      const int b = (v >> a) & 1;
      f[a] = b ? X[a] : __dadd_rn(1.0, -X[a]);
      s[a] = b ? 1.0 : -1.0;
    }
    d[0] = __dmul_rn(s[0], __dmul_rn(f[1], f[2]));
    d[1] = __dmul_rn(s[1], __dmul_rn(f[0], f[2]));
    d[2] = __dmul_rn(s[2], __dmul_rn(f[0], f[1]));
    if (CLAMP)
    {
#pragma unroll
      for (int a = 0; a < 3; ++a) d[a] = clamp_dev(d[a]);
    }
    const double* xv = x + 3 * (int64_t)xd[v];
#pragma unroll
    for (int i = 0; i < 3; ++i)
    {
      const double ci = xv[i];
#pragma unroll
      for (int j = 0; j < 3; ++j) J[i][j] = __dadd_rn(J[i][j], __dmul_rn(ci, d[j]));
    }
  }
}

__device__ __forceinline__ double det_inv3(const double A[3][3], double B[3][3])
{
  const double w0 = diffprod(A[1][1], A[1][2], A[2][1], A[2][2]);
  const double w1 = diffprod(A[1][0], A[1][2], A[2][0], A[2][2]);
  const double w2 = diffprod(A[1][0], A[1][1], A[2][0], A[2][1]);
  const double w3 = diffprod(A[0][0], A[0][1], w1, w0);
  const double det = fma(A[0][2], w2, w3);
  const double r = 1.0 / det;
  B[0][0] = __dmul_rn(w0, r);
  B[1][0] = __dmul_rn(-w1, r);
  B[2][0] = __dmul_rn(w2, r);
  B[0][1] = __dmul_rn(diffprod(A[0][2], A[0][1], A[2][2], A[2][1]), r);
  B[0][2] = __dmul_rn(diffprod(A[0][1], A[0][2], A[1][1], A[1][2]), r);
  B[1][1] = __dmul_rn(diffprod(A[0][0], A[0][2], A[2][0], A[2][2]), r);
  B[1][2] = __dmul_rn(diffprod(A[1][0], A[0][0], A[1][2], A[0][2]), r);
  B[2][1] = __dmul_rn(diffprod(A[2][0], A[0][0], A[2][1], A[0][1]), r);
  B[2][2] = __dmul_rn(diffprod(A[0][0], A[1][0], A[0][1], A[1][1]), r);
  return det;
}

// precompute_geometric_data: GLL points of the element itself, |det| * w, clamped G.
template <typename T>
__global__ void __launch_bounds__(256)
geom_gll_kernel(int n, int64_t ncells, const double* __restrict__ x,
                const int32_t* __restrict__ xdofs, Tables1D tab, T* __restrict__ G6,
                double* __restrict__ dJw)
{
  const int n2 = n * n, nq = n2 * n;
  const int64_t gid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (gid >= ncells * nq) return;
  const int64_t c = gid / nq;
  const int r = (int)(gid - c * nq);
  const int k = r / n2, col = r - k * n2, i = col / n, j = col - i * n;
  const double X[3] = {tab.pts[i], tab.pts[j], tab.pts[k]};
  double J[3][3], K[3][3];
  jacobian_at<true>(x, xdofs + 8 * c, X, J);
  const double det = det_inv3(J, K);
  const double w = __dmul_rn(__dmul_rn(tab.wts[i], tab.wts[j]), tab.wts[k]);
  const double dj = __dmul_rn(fabs(det), w); // precomputation.hpp:95
  dJw[gid] = dj;
  double g[6];
  int m = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = a; b < 3; ++b)
    {
      double s = 0.0; // :99-100, dot() accumulating into zero, k ascending
#pragma unroll
      for (int l = 0; l < 3; ++l) s = __dadd_rn(s, __dmul_rn(__dmul_rn(K[a][l], dj), K[b][l]));
      g[m++] = clamp_dev(s); // :105-107
    }
  // layout [cell][k][pair][col][2]
  T* base = G6 + ((c * n + k) * 3) * (int64_t)n2 * 2;
#pragma unroll
  for (int p = 0; p < 3; ++p)
  {
    base[((int64_t)p * n2 + col) * 2 + 0] = (T)g[2 * p];
    base[((int64_t)p * n2 + col) * 2 + 1] = (T)g[2 * p + 1];
  }
}

// Affine-cell detection, one warp per cell: A = G(q0) / w_q0 at the first point, then every point
// must satisfy |G(q) - w_q A| <= tol * w_q * max|A| entry by entry (the reference's G is
// J^-1 (|det J| w_q) J^-T, precomputation.hpp:95-100: on a parallelepiped J is constant, so G is
// w_q times a constant matrix up to rounding -- unless the absolute-tolerance clamp of :105-107 bit
// at some points only, in which case the cell stays on the general path).
template <typename T>
__global__ void __launch_bounds__(256)
affine_detect_kernel(int n, int64_t ncells, const T* __restrict__ G6, Tables1D tab, double tol,
                     T* __restrict__ Gc, uint8_t* __restrict__ flag)
{
  const int n2 = n * n, nq = n2 * n;
  const int64_t c = blockIdx.x * (int64_t)(blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x % 32;
  if (c >= ncells) return;
  const T* g = G6 + c * (int64_t)nq * 6;
  auto entry = [&](int k, int col, int m) { return (double)g[((int64_t)(k * 3 + m / 2) * n2 + col) * 2 + (m & 1)]; };
  double A[6], amax = 0;
  const double w0 = tab.wts[0] * tab.wts[0] * tab.wts[0];
#pragma unroll
  for (int m = 0; m < 6; ++m)
  {
    A[m] = entry(0, 0, m) / w0;
    amax = fmax(amax, fabs(A[m]));
  }
  bool ok = amax > 0;
  for (int r = lane; r < nq; r += 32)
  {
    const int k = r / n2, col = r - k * n2, i = col / n, j = col - i * n;
    const double w = tab.wts[i] * tab.wts[j] * tab.wts[k];
#pragma unroll
    for (int m = 0; m < 6; ++m) ok = ok && fabs(entry(k, col, m) - w * A[m]) <= tol * w * amax;
  }
  ok = __all_sync(0xffffffffu, ok);
  if (lane == 0)
  {
    flag[c] = ok ? 1 : 0;
#pragma unroll
    for (int m = 0; m < 6; ++m) Gc[c * 6 + m] = (T)A[m];
  }
}

// G[c] *= coeff[c] for every point of cell c (and the per-cell form, when Gc is not NULL)
template <typename T>
__global__ void __launch_bounds__(256)
scale_cells_kernel(int64_t ncells, int per_cell, const double* __restrict__ coeff, T* __restrict__ G6,
                   T* __restrict__ Gc)
{
  const int64_t gid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (gid < ncells * per_cell) G6[gid] = (T)((double)G6[gid] * coeff[gid / per_cell]);
  if (Gc && gid < ncells * 6) Gc[gid] = (T)((double)Gc[gid] * coeff[gid / 6]);
}

// common/precompute.hpp building blocks at arbitrary reference points.
__global__ void __launch_bounds__(256)
jacobian_data_kernel(int nq, int64_t ncells, const double* __restrict__ x,
                     const int32_t* __restrict__ xdofs, const double* __restrict__ points,
                     const double* __restrict__ weights, double* __restrict__ Jout,
                     double* __restrict__ detout, double* __restrict__ Kout,
                     double* __restrict__ Gout)
{
  const int64_t gid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (gid >= ncells * nq) return;
  const int64_t c = gid / nq;
  const int q = (int)(gid - c * nq);
  const double X[3] = {points[3 * q], points[3 * q + 1], points[3 * q + 2]};
  double J[3][3], K[3][3];
  jacobian_at<false>(x, xdofs + 8 * c, X, J);
  const double det = det_inv3(J, K);
  if (Jout)
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b) Jout[gid * 9 + 3 * a + b] = J[a][b];
  if (detout) detout[gid] = det;
  if (Kout)
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b) Kout[gid * 9 + 3 * a + b] = K[a][b];
  if (Gout)
  {
    const double dj = __dmul_rn(det, weights[q]); // precompute.hpp:165 (no fabs)
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b)
      {
        double s = 0.0;
        for (int l = 0; l < 3; ++l) s = __dadd_rn(s, __dmul_rn(K[a][l], K[b][l]));
        Gout[gid * 9 + 3 * a + b] = __dmul_rn(s, dj);
      }
  }
}
} // namespace

extern "C" int wfx_geometry_create(wfx_ctx* ctx, int P, int dtype, int64_t ncells, int64_t npts,
                                   const double* x_host, const int32_t* xdofs_host,
                                   wfx_geom** out)
{
  WFX_API_BEGIN
  if (!ctx || !out) fail("NULL argument");
  if (P < 1 || P + 1 > WFX_MAXN) fail("degree %d out of range", P);
  if (dtype != WFX_F64 && dtype != WFX_F32) fail("unknown dtype %d", dtype);
  if (ncells < 0 || npts < 0) fail("negative size");
  ScopedDevice sd(ctx->device);
  const int n = P + 1, nq = n * n * n;
  auto* g = new wfx_geom;
  std::unique_ptr<wfx_geom> guard(g);
  g->ctx = ctx;
  g->P = P;
  g->n = n;
  g->nq = nq;
  g->dtype = dtype;
  g->ncells = ncells;
  SetupTimer timer("geometry_create");
  for (int64_t i = 0; i < ncells * 8; ++i)
    if (xdofs_host[i] < 0 || xdofs_host[i] >= npts) fail("geometry dofmap entry out of range");
  g->centroid.resize((size_t)ncells * 3);
  for (int64_t c = 0; c < ncells; ++c)
    for (int a = 0; a < 3; ++a)
    {
      double s = 0;
      for (int v = 0; v < 8; ++v) s += x_host[3 * (int64_t)xdofs_host[8 * c + v] + a];
      g->centroid[3 * c + a] = (float)(s / 8);
    }
  timer.lap("checks + centroids");
  if (!std::getenv("WFX_NO_CONNECTIVITY_COORDS")) structured_cell_coords(ncells, npts, xdofs_host, g->cell_ijk);
  timer.lap("connectivity coordinates");
  if (ncells > 0)
  {
    const size_t esz = dtype == WFX_F64 ? 8 : 4;
    WFX_CUDA(cudaMalloc(&g->G6, (size_t)ncells * nq * 6 * esz));
    WFX_CUDA(cudaMalloc((void**)&g->dJw, (size_t)ncells * nq * sizeof(double)));
    DevBuf<double> dx((size_t)npts * 3);
    DevBuf<int32_t> dxd((size_t)ncells * 8);
    dx.upload(x_host, (size_t)npts * 3);
    dxd.upload(xdofs_host, (size_t)ncells * 8);
    Tables1D tab{};
    gll_points_weights(P, tab.pts, tab.wts);
    const int64_t total = ncells * nq;
    const unsigned grid = (unsigned)((total + 255) / 256);
    if (dtype == WFX_F64)
      geom_gll_kernel<double><<<grid, 256>>>(n, ncells, dx.p, dxd.p, tab, (double*)g->G6, g->dJw);
    else
      geom_gll_kernel<float><<<grid, 256>>>(n, ncells, dx.p, dxd.p, tab, (float*)g->G6, g->dJw);
    WFX_CUDA(cudaGetLastError());
    // affine cells
    WFX_CUDA(cudaMalloc(&g->Gc, (size_t)ncells * 6 * esz));
    WFX_CUDA(cudaMalloc((void**)&g->affine, (size_t)ncells));
    const unsigned agrid = (unsigned)((ncells + 7) / 8);
    if (dtype == WFX_F64)
      affine_detect_kernel<double><<<agrid, 256>>>(n, ncells, (const double*)g->G6, tab, 1e-13, (double*)g->Gc, g->affine);
    else
      affine_detect_kernel<float><<<agrid, 256>>>(n, ncells, (const float*)g->G6, tab, 2e-6, (float*)g->Gc, g->affine);
    WFX_CUDA(cudaGetLastError());
    WFX_CUDA(cudaDeviceSynchronize());
    std::vector<uint8_t> fl((size_t)ncells);
    WFX_CUDA(cudaMemcpy(fl.data(), g->affine, (size_t)ncells, cudaMemcpyDeviceToHost));
    for (uint8_t f : fl) g->n_affine += f;
    timer.lap("G, detJ, affine detection");
  }
  *out = guard.release();
  WFX_API_END
}

extern "C" int wfx_geometry_info(wfx_geom* g, int64_t* ncells, int64_t* n_affine)
{
  WFX_API_BEGIN
  if (!g) fail("geom is NULL");
  if (ncells) *ncells = g->ncells;
  if (n_affine) *n_affine = g->n_affine;
  WFX_API_END
}

extern "C" int wfx_geometry_scale_cells(wfx_geom* g, const double* coeff_host)
{
  WFX_API_BEGIN
  if (!g || !coeff_host) fail("NULL argument");
  if (g->ncells == 0) return 0;
  ScopedDevice sd(g->ctx->device);
  for (int64_t c = 0; c < g->ncells; ++c)
    if (!(coeff_host[c] > 0) || !std::isfinite(coeff_host[c])) fail("cell coefficient %lld is not positive and finite", (long long)c);
  DevBuf<double> d((size_t)g->ncells);
  d.upload(coeff_host, (size_t)g->ncells);
  const int per_cell = g->nq * 6;
  const int64_t total = g->ncells * per_cell;
  const unsigned grid = (unsigned)((total + 255) / 256);
  // the operators' private copies hold the same values per cell in another order: the same scaling keeps
  // each one bitwise equal to the reordered scaled G
  std::vector<std::pair<void*, void*>> targets{{g->G6, g->Gc}};
  for (void* p : g->g_copies) targets.push_back({p, nullptr});
  for (const auto& t : targets)
  {
    if (g->dtype == WFX_F64)
      scale_cells_kernel<double><<<grid, 256>>>(g->ncells, per_cell, d.p, (double*)t.first, (double*)t.second);
    else
      scale_cells_kernel<float><<<grid, 256>>>(g->ncells, per_cell, d.p, (float*)t.first, (float*)t.second);
  }
  WFX_CUDA(cudaGetLastError());
  WFX_CUDA(cudaDeviceSynchronize());
  if (g->cell_coeff.empty()) g->cell_coeff.assign((size_t)g->ncells, 1.0);
  for (int64_t c = 0; c < g->ncells; ++c) g->cell_coeff[c] *= coeff_host[c];
  for (wfx_pml* p : g->pmls) pml_scale_cells(p, coeff_host);
  WFX_API_END
}

extern "C" int wfx_geometry_get(wfx_geom* g, double* G_host, double* detJ_host)
{
  WFX_API_BEGIN
  if (!g) fail("geom is NULL");
  ScopedDevice sd(g->ctx->device);
  const int n = g->n, n2 = n * n, nq = g->nq;
  const int64_t nc = g->ncells;
  if (detJ_host && nc)
  {
    std::vector<double> tmp((size_t)nc * nq);
    WFX_CUDA(cudaMemcpy(tmp.data(), g->dJw, tmp.size() * 8, cudaMemcpyDeviceToHost));
    for (int64_t c = 0; c < nc; ++c)
      for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j)
          for (int k = 0; k < n; ++k)
            detJ_host[c * nq + (i * n + j) * n + k] = tmp[c * nq + k * n2 + i * n + j];
  }
  if (G_host && nc)
  {
    const size_t cnt = (size_t)nc * nq * 6;
    std::vector<double> tmp(cnt);
    if (g->dtype == WFX_F64)
      WFX_CUDA(cudaMemcpy(tmp.data(), g->G6, cnt * 8, cudaMemcpyDeviceToHost));
    else
    {
      std::vector<float> t32(cnt);
      WFX_CUDA(cudaMemcpy(t32.data(), g->G6, cnt * 4, cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < cnt; ++i) tmp[i] = t32[i];
    }
    static const int IDX[3][3] = {{0, 1, 2}, {1, 3, 4}, {2, 4, 5}};
    for (int64_t c = 0; c < nc; ++c)
      for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j)
          for (int k = 0; k < n; ++k)
          {
            const int col = g->g_colpos.empty() ? i * n + j : g->g_colpos[i * n + j];
            double* dst = G_host + (c * nq + (i * n + j) * n + k) * 9;
            for (int a = 0; a < 3; ++a)
              for (int b = 0; b < 3; ++b)
              {
                const int m = IDX[a][b];
                dst[3 * a + b] = tmp[(((c * n + k) * 3 + m / 2) * (size_t)n2 + col) * 2 + (m & 1)];
              }
          }
  }
  WFX_API_END
}

extern "C" int wfx_geometry_destroy(wfx_geom* g)
{
  WFX_API_BEGIN
  if (g)
  {
    ScopedDevice sd(g->ctx->device);
    delete g;
  }
  WFX_API_END
}

extern "C" int wfx_compute_jacobian_data(wfx_ctx* ctx, int64_t ncells, int64_t npts,
                                         const double* x_host, const int32_t* xdofs_host, int nq,
                                         const double* points_host, const double* weights_host,
                                         double* J_host, double* detJ_host, double* K_host,
                                         double* G_host)
{
  WFX_API_BEGIN
  if (!ctx) fail("ctx is NULL");
  if (G_host && !weights_host) fail("weights are required to compute G");
  if (ncells <= 0 || nq <= 0) return 0;
  ScopedDevice sd(ctx->device);
  const size_t tot = (size_t)ncells * nq;
  DevBuf<double> dx((size_t)npts * 3), dp((size_t)nq * 3), dw((size_t)nq);
  DevBuf<int32_t> dxd((size_t)ncells * 8);
  dx.upload(x_host, (size_t)npts * 3);
  dxd.upload(xdofs_host, (size_t)ncells * 8);
  dp.upload(points_host, (size_t)nq * 3);
  if (weights_host) dw.upload(weights_host, (size_t)nq);
  DevBuf<double> dJ, dD, dK, dG;
  if (J_host) dJ.alloc(tot * 9);
  if (detJ_host) dD.alloc(tot);
  if (K_host) dK.alloc(tot * 9);
  if (G_host) dG.alloc(tot * 9);
  jacobian_data_kernel<<<(unsigned)((tot + 255) / 256), 256>>>(nq, ncells, dx.p, dxd.p, dp.p, dw.p,
                                                              dJ.p, dD.p, dK.p, dG.p);
  WFX_CUDA(cudaGetLastError());
  WFX_CUDA(cudaDeviceSynchronize());
  if (J_host) dJ.download(J_host, tot * 9);
  if (detJ_host) dD.download(detJ_host, tot);
  if (K_host) dK.download(K_host, tot * 9);
  if (G_host) dG.download(G_host, tot * 9);
  WFX_API_END
}
