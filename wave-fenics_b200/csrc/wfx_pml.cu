// Perfectly matched layer (DESIGN.md section 4.5g): the second-order PML of Grote and Sim (2010) in the weighted form
// of section 4.5e, on the cells where a damping profile zeta_j(x) >= 0 is nonzero.  Per PML dof i and PML cell point q:
//   m~_i (p_tt + sum zeta p_t + sum zeta zeta p + zeta1 zeta2 zeta3 psi)_i = b_i + [D^T phi]_i
//   psi_t = p,   phi_t = -Z phi + a Gamma1 grad w + a Gamma2 grad(psi + s p)
// with a = cK^2 coeff_c, w = p + s p_t the stiffness input of the model (s = 0: w = p) and
//   [D^T phi]_i = -sum_c sum_q grad^ l_i(xi_q) . F_q,   F_q = (|detJ| w)_q J_q^-1 phi_q.
// Two kernels per RK4 stage, launched after the boundary term and before the dense stage update:
//   pml_cell_kernel: one block per PML cell, one thread per point, the cell's w and psi + s p staged in shared memory;
//     writes the cell's D^T phi contribution per point to r [cells][nq] and (UPDATE) steps phi with the RK4 tableau.
//   pml_dof_kernel: one thread per PML dof; sums its r entries in the fixed order of the inverse map, adds them and
//     the diagonal terms to b and (UPDATE) steps psi.
// Both are deterministic (no atomics).  Without a PML nothing here runs.
#include "wfx_internal.h"

#include <algorithm>
#include <cmath>

using namespace wfx;

struct wfx_pml
{
  wfx_ctx* ctx = nullptr;
  wfx_geom* geom = nullptr;
  int P = 0, n = 0, nq = 0, dtype = WFX_F64;
  int64_t ndofs = 0;  // dofs of the mesh
  int64_t ncells = 0; // PML cells
  int64_t npd = 0;    // PML dofs
  double zeta_max = 0;
  std::vector<int32_t> cells;    // geometry cell of each PML cell
  std::vector<int32_t> dofs_h;   // global dof of each PML dof (ascending)
  std::vector<double> coeff;     // composed wfx_geometry_scale_cells coefficient of each PML cell
  DevBuf<double> coeff_d;        // the same on the device
  DevBuf<int32_t> gdm, cdm;      // [ncells][nq] tensor order: global / compact dof
  DevBuf<unsigned char> Kinv;    // [ncells][9][nq] T: J^-1 (entry 3 a + l = dX_a / dx_l)
  DevBuf<unsigned char> djw;     // [ncells][nq] T: |detJ| w
  DevBuf<int32_t> dofs;          // [npd]
  DevBuf<unsigned char> zeta;    // [3][npd] T
  DevBuf<unsigned char> zsum;    // [3][npd] T: sum zeta_j, sum_{j<k} zeta_j zeta_k, zeta1 zeta2 zeta3
  DevBuf<int32_t> inv_off, inv_ent; // PML dof -> entries cell * nq + point of r, ascending
  ~wfx_pml()
  {
    if (geom)
    {
      auto& v = geom->pmls;
      v.erase(std::remove(v.begin(), v.end(), this), v.end());
    }
  }
};

namespace
{
constexpr int PML_NMAX = 9; // P <= 8: the staged arrays of a cell fit the static shared memory in fp64

template <typename T>
struct PmlCellArgs
{
  const int32_t *gdm, *cdm;
  const T *K, *djw, *zeta;
  const double* coeff;
  double cK2;
  T s, bdt, adt;
  int64_t npd;
  const T *w, *u_, *vn;     // stiffness input; p = u_ (stage 0) or w - s vn
  const T *psi_, *psin;      // psi of the stage: psi_ at stage 0, else psin
  T *phi_, *phi0, *phin;     // [cells][3][nq]
  T* r;                      // [cells][nq]
  T D[PML_NMAX * PML_NMAX];  // D[q * N + i] = l_i'(x_q), the stiffness kernels' table
};

// one thread per point: the block is the cell's points rounded up to whole warps
template <int N>
constexpr int pml_block()
{
  return (N * N * N + 31) / 32 * 32;
}

template <typename T, int N, int STAGE, bool UPDATE>
__global__ void __launch_bounds__(pml_block<N>()) pml_cell_kernel(const __grid_constant__ PmlCellArgs<T> a)
{
  constexpr int NQ = N * N * N;
  __shared__ T sW[NQ], sX[NQ], sF[3][NQ];
  const int64_t c = blockIdx.x;
  const int t = threadIdx.x;
  const bool on = t < NQ;
  const int i0 = t / (N * N), i1 = (t / N) % N, i2 = t % N;
  // the arrays do not overlap: restrict lets the compiler move a point's loads ahead of its stores
  T* __restrict__ phi_ = a.phi_;
  T* __restrict__ phi0 = a.phi0;
  T* __restrict__ phin = a.phin;
  const T* phs = (STAGE == 0 ? phi_ : phin) + c * 3 * NQ; // the stage's phi, based on one of the two
  // the point's own data first, so that its loads are in flight with the gathers below
  T k[9], ph[3], ps[3], pb[3], z[3], dj = T(0);
  if (on)
  {
#pragma unroll
    for (int e = 0; e < 9; ++e) k[e] = a.K[(c * 9 + e) * NQ + t];
#pragma unroll
    for (int l = 0; l < 3; ++l)
    {
      const int64_t o = c * 3 * NQ + l * NQ + t;
      ph[l] = phs[l * NQ + t];
      if (UPDATE)
      {
        ps[l] = STAGE == 0 ? ph[l] : phi_[o];
        pb[l] = STAGE == 0 ? ph[l] : (STAGE < 3 ? phi0[o] : T(0));
      }
    }
    dj = a.djw[c * NQ + t];
    const int32_t g = a.gdm[c * NQ + t], j = a.cdm[c * NQ + t];
    if (UPDATE) z[0] = a.zeta[j], z[1] = a.zeta[a.npd + j], z[2] = a.zeta[2 * a.npd + j];
    const T wg = a.w[g];
    sW[t] = wg;
    T chi = STAGE == 0 ? a.psi_[j] : a.psin[j];
    if (a.s != T(0))
    {
      const T p = STAGE == 0 ? a.u_[g] : wg - a.s * a.vn[g];
      chi = chi + a.s * p;
    }
    sX[t] = chi;
  }
  __syncthreads();
  if (on)
  {
#pragma unroll
    for (int d = 0; d < 3; ++d) sF[d][t] = dj * (k[3 * d] * ph[0] + k[3 * d + 1] * ph[1] + k[3 * d + 2] * ph[2]);
    if (UPDATE)
    {
      // reference gradients of w and chi = psi + s p at the point, then physical ones: (grad)_l = sum_a K[a][l] g_a
      T gw[3] = {T(0), T(0), T(0)}, gx[3] = {T(0), T(0), T(0)};
#pragma unroll
      for (int m = 0; m < N; ++m)
      {
        const int o0 = (m * N + i1) * N + i2, o1 = (i0 * N + m) * N + i2, o2 = (i0 * N + i1) * N + m;
        const T d0 = a.D[i0 * N + m], d1 = a.D[i1 * N + m], d2 = a.D[i2 * N + m];
        gw[0] += d0 * sW[o0];
        gw[1] += d1 * sW[o1];
        gw[2] += d2 * sW[o2];
        gx[0] += d0 * sX[o0];
        gx[1] += d1 * sX[o1];
        gx[2] += d2 * sX[o2];
      }
      const T ac = (T)(a.cK2 * a.coeff[c]);
      const T g1[3] = {z[1] + z[2] - z[0], z[0] + z[2] - z[1], z[0] + z[1] - z[2]};
      const T g2[3] = {z[1] * z[2], z[0] * z[2], z[0] * z[1]};
#pragma unroll
      for (int l = 0; l < 3; ++l)
      {
        const T pw = k[l] * gw[0] + k[3 + l] * gw[1] + k[6 + l] * gw[2];
        const T px = k[l] * gx[0] + k[3 + l] * gx[1] + k[6 + l] * gx[2];
        const T kphi = ac * (g1[l] * pw + g2[l] * px) - z[l] * ph[l];
        const int64_t o = c * 3 * NQ + l * NQ + t;
        if (STAGE == 0) phi0[o] = ps[l];
        phi_[o] = kphi * a.bdt + ps[l];
        if (STAGE < 3) phin[o] = kphi * a.adt + pb[l];
      }
    }
  }
  __syncthreads();
  if (on)
  {
    T acc = T(0);
#pragma unroll
    for (int m = 0; m < N; ++m)
      acc += a.D[m * N + i0] * sF[0][(m * N + i1) * N + i2] + a.D[m * N + i1] * sF[1][(i0 * N + m) * N + i2] +
             a.D[m * N + i2] * sF[2][(i0 * N + i1) * N + m];
    a.r[c * NQ + t] = -acc;
  }
}

template <typename T>
struct PmlDofArgs
{
  int64_t npd;
  const int32_t *dofs, *off, *ent;
  const T *r, *m, *zsum;
  T s, bdt, adt;
  const T *w, *u_, *v_, *vn;
  T *psi_, *psi0, *psin;
  T* b;
};

template <typename T, int STAGE, bool UPDATE>
__global__ void __launch_bounds__(256) pml_dof_kernel(const PmlDofArgs<T> a)
{
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= a.npd) return;
  const int32_t g = a.dofs[j];
  T acc = T(0);
  for (int32_t e = a.off[j]; e < a.off[j + 1]; ++e) acc += a.r[a.ent[e]];
  T p, pd;
  if (STAGE == 0)
  {
    p = a.u_[g];
    pd = a.v_[g];
  }
  else
  {
    pd = a.vn[g];
    p = a.w[g] - a.s * pd;
  }
  const T ps = a.psi_[j];
  const T psis = STAGE == 0 ? ps : a.psin[j];
  // loaded before the first store (b and psi might alias as far as the compiler knows)
  const T pb = STAGE == 0 ? ps : (UPDATE && STAGE < 3 ? a.psi0[j] : T(0));
  const T diag = a.zsum[j] * pd + a.zsum[a.npd + j] * p + a.zsum[2 * a.npd + j] * psis;
  a.b[g] = a.b[g] + (acc - a.m[j] * diag);
  if (UPDATE)
  {
    if (STAGE == 0) a.psi0[j] = ps;
    a.psi_[j] = p * a.bdt + ps;
    if (STAGE < 3) a.psin[j] = p * a.adt + pb;
  }
}

template <typename T, int N>
void launch_cell_n(int stage, bool update, int64_t ncells, const PmlCellArgs<T>& a, cudaStream_t st)
{
  const unsigned block = (unsigned)pml_block<N>();
  const unsigned grid = (unsigned)ncells;
  if (!update)
  {
    pml_cell_kernel<T, N, 0, false><<<grid, block, 0, st>>>(a);
    return;
  }
  switch (stage)
  {
  case 0: pml_cell_kernel<T, N, 0, true><<<grid, block, 0, st>>>(a); break;
  case 1: pml_cell_kernel<T, N, 1, true><<<grid, block, 0, st>>>(a); break;
  case 2: pml_cell_kernel<T, N, 2, true><<<grid, block, 0, st>>>(a); break;
  default: pml_cell_kernel<T, N, 3, true><<<grid, block, 0, st>>>(a); break;
  }
}

template <typename T>
void launch_pml(const wfx_pml* pm, const PmlStage& q, cudaStream_t st)
{
  PmlCellArgs<T> ca{};
  ca.gdm = pm->gdm.p;
  ca.cdm = pm->cdm.p;
  ca.K = (const T*)pm->Kinv.p;
  ca.djw = (const T*)pm->djw.p;
  ca.zeta = (const T*)pm->zeta.p;
  ca.coeff = pm->coeff_d.p;
  ca.cK2 = q.cK2;
  ca.s = (T)q.s;
  ca.bdt = (T)q.bdt;
  ca.adt = (T)q.adt;
  ca.npd = pm->npd;
  ca.w = (const T*)q.w;
  ca.u_ = (const T*)q.u_;
  ca.vn = (const T*)q.vn;
  ca.psi_ = (const T*)q.psi_;
  ca.psin = (const T*)q.psin;
  ca.phi_ = (T*)q.phi_;
  ca.phi0 = (T*)q.phi0;
  ca.phin = (T*)q.phin;
  ca.r = (T*)q.r;
  double D[WFX_MAXN * WFX_MAXN];
  deriv_1d(pm->P, D, true);
  for (int e = 0; e < pm->n * pm->n; ++e) ca.D[e] = (T)D[e];
  switch (pm->n)
  {
  case 2: launch_cell_n<T, 2>(q.stage, q.update, pm->ncells, ca, st); break;
  case 3: launch_cell_n<T, 3>(q.stage, q.update, pm->ncells, ca, st); break;
  case 4: launch_cell_n<T, 4>(q.stage, q.update, pm->ncells, ca, st); break;
  case 5: launch_cell_n<T, 5>(q.stage, q.update, pm->ncells, ca, st); break;
  case 6: launch_cell_n<T, 6>(q.stage, q.update, pm->ncells, ca, st); break;
  case 7: launch_cell_n<T, 7>(q.stage, q.update, pm->ncells, ca, st); break;
  case 8: launch_cell_n<T, 8>(q.stage, q.update, pm->ncells, ca, st); break;
  default: launch_cell_n<T, 9>(q.stage, q.update, pm->ncells, ca, st); break;
  }
  WFX_CUDA(cudaGetLastError());
  PmlDofArgs<T> da{};
  da.npd = pm->npd;
  da.dofs = pm->dofs.p;
  da.off = pm->inv_off.p;
  da.ent = pm->inv_ent.p;
  da.r = (const T*)q.r;
  da.m = (const T*)q.m;
  da.zsum = (const T*)pm->zsum.p;
  da.s = (T)q.s;
  da.bdt = (T)q.bdt;
  da.adt = (T)q.adt;
  da.w = (const T*)q.w;
  da.u_ = (const T*)q.u_;
  da.v_ = (const T*)q.v_;
  da.vn = (const T*)q.vn;
  da.psi_ = (T*)q.psi_;
  da.psi0 = (T*)q.psi0;
  da.psin = (T*)q.psin;
  da.b = (T*)q.b;
  const unsigned grid = (unsigned)((pm->npd + 255) / 256);
  if (!q.update) pml_dof_kernel<T, 0, false><<<grid, 256, 0, st>>>(da);
  else
    switch (q.stage)
    {
    case 0: pml_dof_kernel<T, 0, true><<<grid, 256, 0, st>>>(da); break;
    case 1: pml_dof_kernel<T, 1, true><<<grid, 256, 0, st>>>(da); break;
    case 2: pml_dof_kernel<T, 2, true><<<grid, 256, 0, st>>>(da); break;
    default: pml_dof_kernel<T, 3, true><<<grid, 256, 0, st>>>(da); break;
    }
  WFX_CUDA(cudaGetLastError());
}

template <typename T>
void upload_as(DevBuf<unsigned char>& d, const std::vector<double>& h)
{
  std::vector<T> t(h.begin(), h.end());
  d.alloc(t.size() * sizeof(T));
  if (!t.empty()) WFX_CUDA(cudaMemcpy(d.p, t.data(), t.size() * sizeof(T), cudaMemcpyHostToDevice));
}
void upload_dtype(DevBuf<unsigned char>& d, const std::vector<double>& h, int dtype)
{
  if (dtype == WFX_F64) upload_as<double>(d, h);
  else upload_as<float>(d, h);
}
} // namespace

namespace wfx
{
void pml_stage(const wfx_pml* pm, const PmlStage& q, cudaStream_t st)
{
  if (pm->ncells == 0) return;
  NvtxRange r("wfx pml");
  if (pm->dtype == WFX_F64) launch_pml<double>(pm, q, st);
  else launch_pml<float>(pm, q, st);
}

void pml_scale_cells(wfx_pml* pm, const double* coeff_host)
{
  for (size_t c = 0; c < pm->cells.size(); ++c) pm->coeff[c] *= coeff_host[pm->cells[c]];
  pm->coeff_d.upload(pm->coeff);
}

PmlShape pml_shape(const wfx_pml* pm)
{
  PmlShape s;
  s.ctx = pm->ctx;
  s.geom = pm->geom;
  s.dtype = pm->dtype;
  s.ndofs = pm->ndofs;
  s.ncells = pm->ncells;
  s.npd = pm->npd;
  s.nq = pm->nq;
  s.zeta_max = pm->zeta_max;
  s.dofs = &pm->dofs_h;
  return s;
}
} // namespace wfx

extern "C" int wfx_pml_create(wfx_ctx* ctx, wfx_geom* geom, int64_t ndofs, const int32_t* dofmap_host, int64_t npts,
                              const double* x_host, const int32_t* xdofs_host, const double* zeta_host, wfx_pml** out)
{
  WFX_API_BEGIN
  if (!ctx || !geom || !out || !zeta_host || (geom->ncells && (!dofmap_host || !x_host || !xdofs_host)))
    fail("NULL argument");
  if (geom->ctx != ctx) fail("pml: the geometry belongs to another context");
  if (ndofs < 0 || ndofs >= (1ll << 31)) fail("pml: ndofs out of range");
  if (geom->n > PML_NMAX) fail("pml: degree %d above %d is not supported", geom->P, PML_NMAX - 1);
  for (int64_t k = 0; k < 3 * ndofs; ++k)
    if (!std::isfinite(zeta_host[k]) || zeta_host[k] < 0)
      fail("pml: zeta[%lld][%lld] must be finite and not negative", (long long)(k / std::max<int64_t>(ndofs, 1)),
           (long long)(k % std::max<int64_t>(ndofs, 1)));
  ScopedDevice sd(ctx->device);
  auto pm = std::make_unique<wfx_pml>();
  pm->ctx = ctx;
  pm->P = geom->P;
  pm->n = geom->n;
  pm->nq = geom->nq;
  pm->dtype = geom->dtype;
  pm->ndofs = ndofs;
  const int n = pm->n, n2 = n * n, nq = pm->nq;
  const int64_t nc_all = geom->ncells;
  std::vector<int32_t> perm(nq);
  tensor_perm(pm->P, perm.data());
  // PML cells: a positive zeta at any of their points; PML dofs: the dofs of those cells, in ascending order
  std::vector<int32_t> cidx(ndofs, -1);
  std::vector<uint8_t> in_pml(ndofs, 0);
  for (int64_t c = 0; c < nc_all; ++c)
  {
    bool hit = false;
    for (int t = 0; t < nq; ++t)
    {
      const int32_t d = dofmap_host[c * nq + t];
      if (d < 0 || d >= ndofs) fail("pml: dofmap entry %d out of range [0,%lld)", d, (long long)ndofs);
      hit = hit || zeta_host[d] > 0 || zeta_host[ndofs + d] > 0 || zeta_host[2 * ndofs + d] > 0;
    }
    if (!hit) continue;
    pm->cells.push_back((int32_t)c);
    for (int t = 0; t < nq; ++t) in_pml[dofmap_host[c * nq + t]] = 1;
  }
  for (int64_t d = 0; d < ndofs; ++d)
    if (in_pml[d])
    {
      cidx[d] = (int32_t)pm->dofs_h.size();
      pm->dofs_h.push_back((int32_t)d);
    }
  pm->ncells = (int64_t)pm->cells.size();
  pm->npd = (int64_t)pm->dofs_h.size();
  if (pm->ncells * nq >= (1ll << 31)) fail("pml: more than 2^31 layer points");
  const int64_t nc = pm->ncells, npd = pm->npd;
  // tensor-ordered dofmaps of the PML cells and the inverse map (cell, point) ascending
  std::vector<int32_t> gdm((size_t)nc * nq), cdm((size_t)nc * nq), off(npd + 1, 0), ent((size_t)nc * nq);
  for (int64_t c = 0; c < nc; ++c)
    for (int t = 0; t < nq; ++t)
    {
      const int32_t d = dofmap_host[(int64_t)pm->cells[c] * nq + perm[t]];
      gdm[c * nq + t] = d;
      cdm[c * nq + t] = cidx[d];
      off[cidx[d] + 1] += 1;
    }
  for (int64_t j = 0; j < npd; ++j) off[j + 1] += off[j];
  {
    std::vector<int32_t> fill(off.begin(), off.end() - 1);
    for (int64_t e = 0; e < nc * nq; ++e) ent[fill[cdm[e]]++] = (int32_t)e;
  }
  // zeta and its symmetric sums per PML dof
  std::vector<double> z(3 * (size_t)npd), zs(3 * (size_t)npd);
  for (int64_t j = 0; j < npd; ++j)
  {
    const int32_t d = pm->dofs_h[j];
    const double z0 = zeta_host[d], z1 = zeta_host[ndofs + d], z2 = zeta_host[2 * ndofs + d];
    z[j] = z0, z[npd + j] = z1, z[2 * npd + j] = z2;
    zs[j] = z0 + z1 + z2;
    zs[npd + j] = z0 * z1 + z0 * z2 + z1 * z2;
    zs[2 * npd + j] = z0 * z1 * z2;
    pm->zeta_max = std::max({pm->zeta_max, z0, z1, z2});
  }
  // J^-1 at the GLL points (tensor order) of the PML cells, and their |detJ| w from the geometry
  std::vector<double> K, dj((size_t)nc * nq);
  if (nc)
  {
    double pts[WFX_MAXN], wts[WFX_MAXN];
    gll_points_weights(pm->P, pts, wts);
    std::vector<double> X((size_t)nq * 3);
    for (int t = 0; t < nq; ++t)
    {
      X[3 * t] = pts[t / n2];
      X[3 * t + 1] = pts[(t / n) % n];
      X[3 * t + 2] = pts[t % n];
    }
    std::vector<int32_t> xd((size_t)nc * 8);
    for (int64_t c = 0; c < nc; ++c)
      for (int v = 0; v < 8; ++v) xd[c * 8 + v] = xdofs_host[(int64_t)pm->cells[c] * 8 + v];
    std::vector<double> Kq((size_t)nc * nq * 9);
    if (wfx_compute_jacobian_data(ctx, nc, npts, x_host, xd.data(), nq, X.data(), nullptr, nullptr, nullptr,
                                  Kq.data(), nullptr))
      fail("%s", wfx_last_error());
    K.resize(Kq.size());
    for (int64_t c = 0; c < nc; ++c)
      for (int t = 0; t < nq; ++t)
        for (int e = 0; e < 9; ++e) K[(c * 9 + e) * nq + t] = Kq[(c * nq + t) * 9 + e];
    std::vector<double> all((size_t)nc_all * nq);
    WFX_CUDA(cudaMemcpy(all.data(), geom->dJw, all.size() * sizeof(double), cudaMemcpyDeviceToHost));
    for (int64_t c = 0; c < nc; ++c)
      for (int t = 0; t < nq; ++t)
      {
        const int i = t / n2, j = (t / n) % n, k = t % n;
        dj[c * nq + t] = all[(int64_t)pm->cells[c] * nq + k * n2 + i * n + j];
      }
  }
  pm->coeff.assign((size_t)nc, 1.0);
  if (!geom->cell_coeff.empty())
    for (int64_t c = 0; c < nc; ++c) pm->coeff[c] = geom->cell_coeff[pm->cells[c]];
  pm->coeff_d.upload(pm->coeff);
  pm->gdm.upload(gdm);
  pm->cdm.upload(cdm);
  pm->inv_off.upload(off);
  pm->inv_ent.upload(ent);
  pm->dofs.upload(pm->dofs_h);
  upload_dtype(pm->Kinv, K, pm->dtype);
  upload_dtype(pm->djw, dj, pm->dtype);
  upload_dtype(pm->zeta, z, pm->dtype);
  upload_dtype(pm->zsum, zs, pm->dtype);
  // scaled with the geometry from now on (wfx_geometry_scale_cells)
  pm->geom = geom;
  geom->pmls.push_back(pm.get());
  *out = pm.release();
  WFX_API_END
}

extern "C" int wfx_pml_info(wfx_pml* pml, int64_t* ncells, int64_t* ndofs, double* zeta_max)
{
  WFX_API_BEGIN
  if (!pml) fail("pml is NULL");
  if (ncells) *ncells = pml->ncells;
  if (ndofs) *ndofs = pml->npd;
  if (zeta_max) *zeta_max = pml->zeta_max;
  WFX_API_END
}

extern "C" int wfx_pml_destroy(wfx_pml* pml)
{
  WFX_API_BEGIN
  if (pml)
  {
    ScopedDevice sd(pml->ctx->device);
    delete pml;
  }
  WFX_API_END
}
