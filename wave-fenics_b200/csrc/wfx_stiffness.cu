// Sum-factorised stiffness apply  y (+)= -c0^2 K x  on GLL hexahedra.
// Replaces StiffnessOperator::operator() + skernel (common/operators.hpp:113-133,183-200),
// whose dense 2*3*nq*nd MAC loop per cell becomes three 1-D contractions with the GLL
// derivative matrix per direction (SURVEY.md App. A.9), and the gather -> kernel -> atomic
// scatter chain of the hackathon GPU operators (common/cuda/mass.hpp:76-95,
// common/cuda/scatter.cu:38-45), which becomes one kernel with an atomic-free scatter.
//
// Thread mapping: the N^2 threads of a cell each own one grid line per direction ("three
// roles", see cell_part1); a 1-D contraction is register-only with the derivative matrix in the
// kernel-parameter constant bank, lines are exchanged through two shared tiles transformed in
// place.  G (symmetric, 6 entries per point) streams from HBM exactly once as 128-bit loads,
// software-prefetched into registers one cell ahead and into L2 (bulk prefetch) one more.
//
// Kernels:
//   stiff_cell_kernel       simple: cells coloured, global gather / read-modify-write scatter
//   stiff_brick_kernel      product path: one CTA per batch of cells (wfx_plan.h); batch dofs
//                           staged in shared memory, each written back once; optional fused
//                           diagonal scaling (the lumped-mass inverse) on the LAST touch; colours
//                           are consecutive launches chained by programmatic dependent launch.
//                           REG = every batch is a lattice brick: arithmetic shared-memory
//                           positions, no staged local dofmap.
//   stiff_cell2_kernel      streamed cells: no dof arrays in shared memory, x gathered and y updated
//                           in global memory, FIRST / LAST flags in the per-point dofmap (fused scaling,
//                           no memset), cells in colour order or in the order of a brick plan with a
//                           round barrier; WFX_STIFF_AUTO takes it where it measured faster (P7 fp32).
// (A persistent single-launch form of the brick kernel was measured slower and removed:
//  DESIGN.md section 6.)
#include "wfx_internal.h"
#include "wfx_plan.h"

#include <algorithm>
#include <type_traits>
#include <cstdlib>
#include <cstring>

using namespace wfx;

namespace
{
template <typename T> struct Vec2;
template <> struct Vec2<double> { using type = double2; };
template <> struct Vec2<float> { using type = float2; };

// streaming (read-once) 2-element global load that does not allocate in L1
__device__ __forceinline__ double2 ld_stream(const double2* p)
{
  double2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ float2 ld_stream(const float2* p)
{
  float2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  return r;
}

// read-once scalar loads that leave L1 to the loads in flight (L1 is the landing buffer of the
// G stream: its capacity bounds the bytes in flight per SM, see DESIGN.md)
__device__ __forceinline__ uint32_t ld_once(const uint32_t* p)
{
  uint32_t r;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ double ld_once(const double* p)
{
  double r;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ float ld_once(const float* p)
{
  float r;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// asynchronous global -> shared copy of one scalar (LDGSTS): no register staging, no stall at issue
__device__ __forceinline__ void cp_async_scalar(double* dst_smem, const double* src)
{
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_scalar(float* dst_smem, const float* src)
{
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// fire-and-forget prefetch of a contiguous block into L2 (bytes multiple of 16, one request)
__device__ __forceinline__ void l2_prefetch_bulk(const void* p, uint32_t bytes)
{
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
#ifndef WFX_PF_DIST
#define WFX_PF_DIST 1 // measured at 64^3 P4 fp64: 1 -> 0.604 ms, 2 -> 0.619, 3 -> 0.631, 4 -> 0.650, none -> 0.695
#endif
constexpr int PF_DIST = WFX_PF_DIST; // rounds the L2 prefetch of G runs ahead of the register loads
// one-shot TMA bulk copy global -> shared with mbarrier completion (bytes multiple of 16)
__device__ __forceinline__ void bulk_copy_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
  uint32_t done = 0;
  while (!done)
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Checked build (-DWFX_CHECKED): device-side bounds checks on every index the kernels form -- the
// pool's compute-sanitizer is closed, so the memory-safety evidence comes from running the GPU test
// suite against this build (profiles/r2_checked_build.md).  A violation prints and traps.
#ifdef WFX_CHECKED
#define WFX_DEV_ASSERT(cond)                                                                          \
  do                                                                                                  \
  {                                                                                                   \
    if (!(cond))                                                                                      \
    {                                                                                                 \
      printf("wfx check failed: %s (%s:%d) block %d thread %d\n", #cond, __FILE__, __LINE__,         \
             (int)blockIdx.x, (int)threadIdx.x);                                                      \
      __trap();                                                                                       \
    }                                                                                                 \
  } while (0)
#else
#define WFX_DEV_ASSERT(cond) ((void)0)
#endif

#ifndef WFX_PERSIST_UW
#define WFX_PERSIST_UW 11
#endif
#ifndef WFX_PERSISTENT_DEFAULT
#define WFX_PERSISTENT_DEFAULT 0
#endif

template <int N> struct Cfg; // per-degree launch configuration (below)

template <typename T, int N>
struct DMat
{
  T d[N * N]; // D[q*N+i] = l_i'(x_q), [0,1,interior] ordering, clamped
  T w[N];     // 1-D GLL weights (affine fast path: G(q) = w_i w_j w_k * A_cell)
};

// Optional phase timer (build with -DWFX_TIMING): lane 0 of every warp accumulates the
// cycles spent between marks; no-op otherwise.
#ifdef WFX_TIMING
__device__ long long* g_wfx_timing = nullptr;
struct PhaseTimer
{
  long long acc[12], last;
  bool on;
  __device__ void start(bool lane0) { on = lane0; for (int q = 0; q < 12; ++q) acc[q] = 0; last = clock64(); }
  __device__ __forceinline__ void mark(int ph) { if (on) { long long t = clock64(); acc[ph] += t - last; last = t; } }
  __device__ void flush(int gwarp) { if (on && g_wfx_timing) for (int q = 0; q < 12; ++q) g_wfx_timing[(long long)gwarp * 12 + q] = acc[q]; }
};
#else
struct PhaseTimer
{
  __device__ __forceinline__ void start(bool) {}
  __device__ __forceinline__ void mark(int) {}
  __device__ __forceinline__ void flush(int) {}
};
#endif

struct WarpSync
{
  __device__ __forceinline__ void operator()() const { __syncwarp(); }
};
struct BlockSync
{
  __device__ __forceinline__ void operator()() const { __syncthreads(); }
};

// Shared-memory tiles of one cell slot: A [k][i][j] and AT [k][j][i], with plane strides and
// row offsets chosen so that every access pattern of the three roles below is free of bank
// conflicts for 64-bit words (16 banks of 8 bytes per half-warp).  For N = 5 the layout was
// found by search (rows of AT at offsets {0,20,7,26,13} inside a 33-word plane); other
// degrees use the plain layout.
// RS = stride between the rows of a plane (WB = bytes per word).  Roles J / I have every lane walk its
// own row, so lane l reads word l * RS + m: for 64-bit words RS is odd -- an even RS folds the 16 lanes
// of a half-warp onto a few banks (N = 8 unpadded: two banks, every row access an 8-way conflict;
// measured P7 fp64 0.644 -> 0.579 ms).  32-bit rows stay unpadded: the compiler reads them with 128-bit
// loads, and both an odd stride (P7 fp32 0.311 -> 0.323 ms) and a 12-word stride that keeps the
// alignment (0.329 ms) measured slower.
template <int N, int WB = 8>
struct Tiles
{
#ifndef WFX_NO_ROW_PAD
  static constexpr int RS = (WB == 8 && N % 2 == 0) ? N + 1 : N;
#else
  static constexpr int RS = N;
#endif
  static constexpr int PS_A = N * RS, PS_T = N * RS;
  __host__ __device__ static constexpr int boff(int j) { return j * RS; }
};
template <int WB>
struct Tiles<5, WB>
{
  static constexpr int RS = 5;
  static constexpr int PS_A = 25, PS_T = 33;
  __host__ __device__ static constexpr int boff(int j)
  {
    return j == 0 ? 0 : (j == 1 ? 20 : (j == 2 ? 7 : (j == 3 ? 26 : 13)));
  }
};
template <int N, int WB> __host__ __device__ constexpr int slot_elems() { return N * (Tiles<N, WB>::PS_A + Tiles<N, WB>::PS_T); }
template <int N> __host__ __device__ constexpr int ndp_of() { return (N * N * N + 7) & ~7; } // ldm slot stride

// per-thread tile offsets of the three roles (constant for the whole kernel)
struct RoleOff
{
  int kA, kT; // role K: element (k) of this thread's column is A[k*PS_A + kA], AT[k*PS_T + kT]
  int rA, rT; // roles J / I: this thread's row starts at A[rA], AT[rT]
  int colK;   // role K: i*N + j (column of G6 and of the local dofmap)
  int iK, jK, kJ, iJ, kI, jI; // the lines this thread owns in the three roles
};
template <int N, int WB>
__device__ __forceinline__ RoleOff role_offsets(int lane)
{
  using TL = Tiles<N, WB>;
  const int hi = lane / N, lo = lane % N;
  RoleOff o;
  o.kA = hi * TL::RS + lo;                  // role K: i = hi, j = lo
  o.kT = TL::boff(lo) + hi;
  o.rA = hi * TL::PS_A + lo * TL::RS;       // role J: k = hi, i = lo, row over j
  o.rT = hi * TL::PS_T + TL::boff(lo);      // role I: k = hi, j = lo, row over i
  o.colK = lane;
  o.iK = hi, o.jK = lo, o.kJ = hi, o.iJ = lo, o.kI = hi, o.jI = lo;
  return o;
}

// Layout policies: tile geometry + the lane -> line maps of the three roles.
// LayoutStd: lane = hi*N + lo in all roles, rows stored in index order.
template <int N, int WB>
struct LayoutStd
{
  static constexpr int PS_A = Tiles<N, WB>::PS_A, PS_T = Tiles<N, WB>::PS_T;
  static constexpr int AT_OFF = N * PS_A, SLOT_ELEMS = N * (PS_A + PS_T);
  __host__ __device__ static constexpr int eA(int n) { return n; } // offset of element j = n in a row of A
  __host__ __device__ static constexpr int eT(int n) { return n; } // offset of element i = n in a row of AT
  __device__ static __forceinline__ RoleOff offsets(int lane) { return role_offsets<N, WB>(lane); }
};

// LayoutP4D: degree 4, 64-bit words, regular bricks whose lattice strides are Sx = 5, Sy = 2
// (mod 16).  Found by tools/bank_layout_search.py: with these lane maps every shared-memory
// access of a cell -- the dof lines of roles K and J, the y accumulation, all tile rows and
// columns -- is free of bank conflicts; role I's dof line costs 3 wavefronts instead of 2 (no
// stride triple makes all three roles conflict-free).  Rows are 5 words at 5*a(.) inside a
// 33-word plane, a() = ascending lattice position; row elements are permuted (eA / eT).
__device__ __constant__ uint8_t c_p4d_lanes[6][25] = {
    // role K lane -> i, j
    {2, 2, 2, 3, 4, 4, 4, 3, 3, 0, 0, 1, 2, 2, 3, 3, 0, 0, 1, 1, 0, 4, 4, 1, 1},
    {3, 4, 1, 3, 0, 2, 3, 4, 1, 3, 4, 3, 0, 2, 0, 2, 0, 2, 0, 2, 1, 4, 1, 4, 1},
    // role J lane -> k, i
    {0, 2, 3, 4, 1, 0, 2, 3, 4, 1, 0, 2, 3, 4, 1, 0, 2, 3, 4, 1, 0, 2, 3, 4, 1},
    {0, 0, 0, 0, 0, 2, 2, 2, 2, 2, 3, 3, 3, 3, 3, 4, 4, 4, 4, 4, 1, 1, 1, 1, 1},
    // role I lane -> k, j
    {4, 0, 2, 3, 4, 1, 0, 1, 3, 3, 4, 2, 0, 2, 3, 2, 0, 2, 4, 0, 1, 1, 3, 4, 1},
    {2, 3, 3, 3, 3, 3, 4, 4, 4, 0, 0, 4, 2, 2, 2, 1, 0, 0, 4, 1, 0, 1, 1, 1, 2}};
struct LayoutP4D
{
  static constexpr int N = 5, PS_A = 33, PS_T = 33;
  static constexpr int AT_OFF = N * PS_A, SLOT_ELEMS = N * (PS_A + PS_T);
  static constexpr int SX_MOD = 5, SY_MOD = 2; // required lattice strides modulo 16
  __host__ __device__ static constexpr int eA(int n) { return n == 0 ? 3 : n == 1 ? 2 : n == 2 ? 4 : n == 3 ? 0 : 1; }
  __host__ __device__ static constexpr int eT(int n) { return n == 0 ? 0 : n == 1 ? 2 : n == 2 ? 1 : n; }
  __host__ __device__ static constexpr int a(int q) { return q == 0 ? 0 : (q == 1 ? N - 1 : q - 1); }
  __device__ static __forceinline__ RoleOff offsets(int lane)
  {
    RoleOff o;
    o.iK = c_p4d_lanes[0][lane], o.jK = c_p4d_lanes[1][lane];
    o.kJ = c_p4d_lanes[2][lane], o.iJ = c_p4d_lanes[3][lane];
    o.kI = c_p4d_lanes[4][lane], o.jI = c_p4d_lanes[5][lane];
    o.colK = o.iK * N + o.jK;
    o.kA = 5 * a(o.iK) + eA(o.jK);
    o.kT = 5 * a(o.jK) + eT(o.iK);
    o.rA = o.kJ * PS_A + 5 * a(o.iJ);
    o.rT = o.kI * PS_T + 5 * a(o.jI);
    return o;
  }
};
// column position of point (i,j) in a G6 whose columns were reordered to LayoutP4D's role K lanes
__device__ __constant__ uint8_t c_p4d_colpos[25] = {16, 20, 17, 9, 10, 18, 24, 19, 11, 23, 12, 2, 13,
                                                    0,  1,  14, 8, 15, 3,  7,  4,  22, 5,  6, 21};
const uint8_t h_p4d_colpos[25] = {16, 20, 17, 9, 10, 18, 24, 19, 11, 23, 12, 2, 13,
                                  0,  1,  14, 8, 15, 3,  7,  4,  22, 5,  6, 21};
// G6 column this thread loads in role K (g_order: 0 = columns by i*N+j, 1 = LayoutP4D lane order)
template <typename L, int N>
__device__ __forceinline__ int g_column(const RoleOff& ro, int lane, int g_order)
{
  if constexpr (N == 5)
  {
    if (g_order) return std::is_same<L, LayoutP4D>::value ? lane : (int)c_p4d_colpos[ro.colK];
  }
  return ro.colK;
}

// G of one cell for this thread's column: [k][pair] 2-vectors, streamed once from HBM.  The
// registers hold a window of GW planes (GW = N: the whole cell); this loads the first GW.
template <typename T, int N, int GW>
__device__ __forceinline__ void load_G(const T* __restrict__ Gc, int col,
                                       typename Vec2<T>::type (&g)[GW][3])
{
  using V2 = typename Vec2<T>::type;
  const V2* gp = reinterpret_cast<const V2*>(Gc) + col;
#pragma unroll
  for (int k = 0; k < GW; ++k)
#pragma unroll
    for (int p = 0; p < 3; ++p) g[k][p] = ld_stream(gp + (k * 3 + p) * (N * N));
}

// Sum-factorised cell kernel, "one line per thread, three roles".  Each of the N^2 threads
// of a cell (lane = hi*N + lo) plays three roles, owning a full grid line in registers:
//    role K: points (i=hi, j=lo, k=*)   -- the gather/scatter role, holds u, G, f, y
//    role J: points (k=hi, i=lo, j=*)
//    role I: points (k=hi, j=lo, i=*)
// A 1-D contraction along a line is register-only and its derivative-matrix operand is a
// compile-time index into the kernel-parameter constant bank (no registers, no shared
// memory for D).  Lines move between roles through two shared tiles, transformed IN PLACE:
// role K writes A [k][i][j] and AT [k][j][i]; role J reads its row of A, contracts it and
// writes the result over the same row (it is the row's only reader); role I does the same
// with its row of AT; role K reads its column back.
// Part 1:  w0 = sum_m D[i][m] u(m,j,k), w1 = sum_m D[j][m] u(i,m,k), w2 = sum_m D[k][m] u(i,j,m),
//          f = coeff * G w   (SURVEY.md App. A.9); f0 -> AT, f1 -> A, f2 stays in registers.
// Part 2:  y(i,j,k) = sum_m D[m][i] f0(m,j,k) + D[m][j] f1(i,m,k) + D[m][k] f2(i,j,m).
// Inactive threads (padding lanes / empty slots) only take part in the synchronisation.
// L: layout policy; ROW_A: the row belongs to tile A (elements by j) or AT (elements by i)
template <typename T, int N, bool TRANSPOSE, typename L, bool ROW_A>
__device__ __forceinline__ void line_transform(T* __restrict__ row, const DMat<T, N>& Dm)
{
  T l[N], o[N];
#pragma unroll
  for (int m = 0; m < N; ++m) l[m] = row[ROW_A ? L::eA(m) : L::eT(m)];
#pragma unroll
  for (int n = 0; n < N; ++n)
  {
    T s = 0;
#pragma unroll
    for (int m = 0; m < N; ++m) s += (TRANSPOSE ? Dm.d[m * N + n] : Dm.d[n * N + m]) * l[m];
    o[n] = s;
  }
#pragma unroll
  for (int n = 0; n < N; ++n) row[ROW_A ? L::eA(n) : L::eT(n)] = o[n];
}

// second half of part 1: w2 from the register line, w0 / w1 from the tiles, f = coeff * G w
// The G registers are a rotating window of GW planes over the stream "cell, next cell, ...":
// as soon as plane k is consumed its slot is refilled with the plane GW positions further on
// (gcur: this cell, gnext: the next one, nullable), so the loads of a cell are spread over the
// phase instead of hitting the load pipe (and L1, their landing buffer) in one burst.  GW = N keeps
// a whole cell in flight (P <= 4); the higher degrees hold fewer planes to stay inside the register
// budget and lean on the L2 prefetch for latency.  N is padded to a multiple of GW with planes that
// are never loaded, which keeps every slot index a compile-time constant.
template <typename T, int N, typename L, int GW>
__device__ __forceinline__ void g_multiply(const T (&u)[N], typename Vec2<T>::type (&g)[GW][3],
                                           T* __restrict__ A, T* __restrict__ AT, const RoleOff& ro,
                                           const DMat<T, N>& Dm, T coeff, T (&f2)[N],
                                           const typename Vec2<T>::type* gcur,
                                           const typename Vec2<T>::type* gnext)
{
  constexpr int NP = ((N + GW - 1) / GW) * GW;
  constexpr int NPW = NP;
#pragma unroll
  for (int k = 0; k < NP; ++k)
  {
    if (k < N)
    {
      T w2 = 0;
#pragma unroll
      for (int m = 0; m < N; ++m) w2 += Dm.d[k * N + m] * u[m];
      const T w0 = AT[k * L::PS_T + ro.kT];
      const T w1 = A[k * L::PS_A + ro.kA];
      const T g00 = g[k % GW][0].x, g01 = g[k % GW][0].y, g02 = g[k % GW][1].x;
      const T g11 = g[k % GW][1].y, g12 = g[k % GW][2].x, g22 = g[k % GW][2].y;
      AT[k * L::PS_T + ro.kT] = coeff * (g00 * w0 + g01 * w1 + g02 * w2); // f0
      A[k * L::PS_A + ro.kA] = coeff * (g01 * w0 + g11 * w1 + g12 * w2);  // f1
      f2[k] = coeff * (g02 * w0 + g12 * w1 + g22 * w2);
    }
    const int t = k + GW;
    if (t < N)
    {
      if (gcur)
      {
#pragma unroll
        for (int p = 0; p < 3; ++p) g[k % GW][p] = ld_stream(gcur + (t * 3 + p) * (N * N));
      }
    }
    else if (t >= NPW && t - NPW < N)
    {
      if (gnext)
      {
#pragma unroll
        for (int p = 0; p < 3; ++p) g[k % GW][p] = ld_stream(gnext + ((t - NPW) * 3 + p) * (N * N));
      }
    }
  }
}

// Affine cells: G(q) = w_q A with one symmetric A per cell (ga: 00,01,02,11,12,22) and
// csk[k] = coeff * w_i w_j w_k for this thread's column -- no per-point G is read.
template <typename T, int N, typename L>
__device__ __forceinline__ void g_multiply_affine(const T (&u)[N], const T (&ga)[6], const T (&csk)[N],
                                                  T* __restrict__ A, T* __restrict__ AT, const RoleOff& ro,
                                                  const DMat<T, N>& Dm, T (&f2)[N])
{
#pragma unroll
  for (int k = 0; k < N; ++k)
  {
    T w2 = 0;
#pragma unroll
    for (int m = 0; m < N; ++m) w2 += Dm.d[k * N + m] * u[m];
    const T w0 = AT[k * L::PS_T + ro.kT];
    const T w1 = A[k * L::PS_A + ro.kA];
    AT[k * L::PS_T + ro.kT] = csk[k] * (ga[0] * w0 + ga[1] * w1 + ga[2] * w2); // f0
    A[k * L::PS_A + ro.kA] = csk[k] * (ga[1] * w0 + ga[3] * w1 + ga[4] * w2);  // f1
    f2[k] = csk[k] * (ga[2] * w0 + ga[4] * w1 + ga[5] * w2);
  }
}

template <typename T, int N, typename L, int GW, typename Sync>
__device__ __forceinline__ void cell_part1(const T (&u)[N], typename Vec2<T>::type (&g)[GW][3],
                                           T* __restrict__ tiles, const RoleOff& ro,
                                           const DMat<T, N>& Dm, T coeff, bool active, Sync sync,
                                           T (&f2)[N], PhaseTimer& tm,
                                           const typename Vec2<T>::type* gcur = nullptr,
                                           const typename Vec2<T>::type* gnext = nullptr)
{
  T* A = tiles;
  T* AT = tiles + L::AT_OFF;
  if (active)
  {
#pragma unroll
    for (int k = 0; k < N; ++k)
    {
      A[k * L::PS_A + ro.kA] = u[k];
      AT[k * L::PS_T + ro.kT] = u[k];
    }
  }
  sync();
  tm.mark(1);
  if (active)
  {
    line_transform<T, N, false, L, true>(A + ro.rA, Dm);   // u(i, ., k) -> w1(i, ., k)
    line_transform<T, N, false, L, false>(AT + ro.rT, Dm); // u(., j, k) -> w0(., j, k)
  }
  sync();
  tm.mark(2);
  if (active) g_multiply<T, N, L, GW>(u, g, A, AT, ro, Dm, coeff, f2, gcur, gnext);
  tm.mark(3);
}

// Part 1 when all three roles already hold their input line (regular bricks: the lines are
// read straight from the batch's staged dofs): no tile round trip for u and one barrier less.
template <typename T, int N, typename L, int GW, typename Sync>
__device__ __forceinline__ void cell_part1_reg(const T (&u)[N], const T (&lj)[N], const T (&lI)[N],
                                               typename Vec2<T>::type (&g)[GW][3],
                                               T* __restrict__ tiles, const RoleOff& ro,
                                               const DMat<T, N>& Dm, T coeff, bool active, Sync sync,
                                               T (&f2)[N], PhaseTimer& tm,
                                               const typename Vec2<T>::type* gcur = nullptr,
                                               const typename Vec2<T>::type* gnext = nullptr)
{
  T* A = tiles;
  T* AT = tiles + L::AT_OFF;
  tm.mark(1);
  if (active)
  {
#pragma unroll
    for (int n = 0; n < N; ++n)
    {
      T s1 = 0, s0 = 0;
#pragma unroll
      for (int m = 0; m < N; ++m)
      {
        s1 += Dm.d[n * N + m] * lj[m];
        s0 += Dm.d[n * N + m] * lI[m];
      }
      A[ro.rA + L::eA(n)] = s1;  // w1(i, n, k)
      AT[ro.rT + L::eT(n)] = s0; // w0(n, j, k)
    }
  }
  sync();
  tm.mark(2);
  if (active) g_multiply<T, N, L, GW>(u, g, A, AT, ro, Dm, coeff, f2, gcur, gnext);
  tm.mark(3);
}

template <typename T, int N, typename L, typename Sync>
__device__ __forceinline__ void cell_part1_reg_affine(const T (&u)[N], const T (&lj)[N], const T (&lI)[N],
                                                      const T (&ga)[6], const T (&csk)[N],
                                                      T* __restrict__ tiles, const RoleOff& ro,
                                                      const DMat<T, N>& Dm, bool active, Sync sync,
                                                      T (&f2)[N], PhaseTimer& tm)
{
  T* A = tiles;
  T* AT = tiles + L::AT_OFF;
  tm.mark(1);
  if (active)
  {
#pragma unroll
    for (int n = 0; n < N; ++n)
    {
      T s1 = 0, s0 = 0;
#pragma unroll
      for (int m = 0; m < N; ++m)
      {
        s1 += Dm.d[n * N + m] * lj[m];
        s0 += Dm.d[n * N + m] * lI[m];
      }
      A[ro.rA + L::eA(n)] = s1;  // w1(i, n, k)
      AT[ro.rT + L::eT(n)] = s0; // w0(n, j, k)
    }
  }
  sync();
  tm.mark(2);
  if (active) g_multiply_affine<T, N, L>(u, ga, csk, A, AT, ro, Dm, f2);
  tm.mark(3);
}

template <typename T, int N, typename L, typename Sync>
__device__ __forceinline__ void cell_part2(const T (&f2)[N], T* __restrict__ tiles, const RoleOff& ro,
                                           const DMat<T, N>& Dm, bool active, Sync sync, T (&yv)[N],
                                           PhaseTimer& tm)
{
  T* A = tiles;
  T* AT = tiles + L::AT_OFF;
  sync(); // f0 / f1 visible
  if (active)
  {
    line_transform<T, N, true, L, true>(A + ro.rA, Dm);   // f1(i, ., k) -> sum_m D[m][.] f1(i,m,k)
    line_transform<T, N, true, L, false>(AT + ro.rT, Dm); // f0(., j, k) -> sum_m D[m][.] f0(m,j,k)
  }
  sync();
  tm.mark(5);
  if (active)
  {
#pragma unroll
    for (int k = 0; k < N; ++k)
    {
      T s = AT[k * L::PS_T + ro.kT] + A[k * L::PS_A + ro.kA];
#pragma unroll
      for (int m = 0; m < N; ++m) s += Dm.d[m * N + k] * f2[m];
      yv[k] = s;
    }
  }
}

// ---- simple kernel: coloured cells, global gather / scatter -----------------------
template <typename T, int N, int SLOT, int CPB>
__global__ void __launch_bounds__(SLOT* CPB)
stiff_cell_kernel(const int32_t* __restrict__ cells, int ncl, const int32_t* __restrict__ tdm,
                  const T* __restrict__ G6, const T* __restrict__ x, T* __restrict__ y,
                  const DMat<T, N> Dm, T coeff, int g_order)
{
  constexpr int N2 = N * N, ND = N2 * N;
  using V2 = typename Vec2<T>::type;
  __shared__ __align__(16) T s_w[CPB][slot_elems<N, sizeof(T)>()];
  const int slot = threadIdx.x / SLOT, col = threadIdx.x % SLOT;
  const int ci = blockIdx.x * CPB + slot;
  const bool active = (col < N2) && (ci < ncl);
  const int64_t cell = active ? cells[ci] : 0;
  const RoleOff ro = role_offsets<N, sizeof(T)>(active ? col : 0);
  int32_t dof[N];
  T u[N], yv[N], f2[N];
  V2 g[N][3];
#pragma unroll
  for (int k = 0; k < N; ++k)
  {
    dof[k] = active ? tdm[cell * ND + k * N2 + col] : 0;
    u[k] = active ? x[dof[k]] : T(0);
    yv[k] = 0;
  }
  if (active) load_G<T, N, N>(G6 + cell * (int64_t)(6 * ND), g_column<LayoutStd<N, sizeof(T)>, N>(ro, col, g_order), g);
  PhaseTimer tm;
  tm.start(false);
  cell_part1<T, N, LayoutStd<N, sizeof(T)>, N>(u, g, s_w[slot], ro, Dm, coeff, active, BlockSync(), f2, tm);
  cell_part2<T, N, LayoutStd<N, sizeof(T)>>(f2, s_w[slot], ro, Dm, active, BlockSync(), yv, tm);
  if (active)
  {
#pragma unroll
    for (int k = 0; k < N; ++k) y[dof[k]] += yv[k];
  }
}

// ---- streamed-cell kernel: coloured cells, no shared-memory dof arrays ------------------------
// At high degree a batch of the brick kernel degenerates: a 2x2x2 brick of P7 cells already fills
// the shared memory two CTAs can have, its eight cells all touch each other (W = 1, one cell at a
// time) and an SM ends up with six warps.  Per cell, though, there is plenty of work (N^3 points) and
// little sharing (N^3 points on (N-1)^3 dofs), so the dofs need not be staged at all: cells are
// coloured (no two cells of a colour share a dof), a slot of SLOT threads walks `cps` consecutive
// cells of its colour, gathers x straight from global memory, and updates y with a plain
// read-modify-write.  What the brick kernel gets from its batch arrays is recovered with flags in the
// per-point dofmap: FIRST (lowest colour touching the dof: overwrite, no memset, no read of y) and
// LAST (highest colour: apply the fused diagonal scaling), so the fused stiffness + mass apply is
// still one pass.  Software pipeline of a slot: the next cell's dof indices are loaded a cell ahead,
// its x values are gathered into the registers of u as soon as the G multiply has consumed u, its G
// planes roll into the register window inside the G multiply (g_multiply) and the cell after that
// goes to L2 by bulk prefetch.  Colours are consecutive launches chained by programmatic dependent
// launch; only the first access to y waits for the previous colour.
template <typename T>
struct Cell2Args
{
  const int32_t* cells;  // cell ids sorted by colour
  const uint32_t* tdmf;  // [ncells][ND] k-major point order: global dof | BD_FIRST | BD_LAST
  const T* G6;
  const T* x;
  T* y;
  const T* scale; // nullable: applied on the LAST touch of a dof
  T coeff;
  int beta;    // 0: FIRST touch overwrites y; 1: accumulates into y
  int g_order; // column order of G6 (see g_column)
  int cps;     // cells per slot (colour-ordered form)
  int64_t ndofs, ncells;
  // brick-ordered form (BRICK): one CTA per batch of the brick plan, one iteration per round
  const int32_t* round_off; // [nbatches+1]
  const int32_t* slot_cell; // [nrounds_total*CPB] cell id or -1
  int uni_nr;               // > 0: every batch has this many rounds
};

struct SlotBarSync
{
  int id, nthr; // named barrier of the slot's warps (id 0 is __syncthreads)
  __device__ __forceinline__ void operator()() const
  {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthr) : "memory");
  }
};

// BRICK: the cells come in the order of the brick plan instead -- one CTA per batch (a spatially
// compact brick of cells), iteration r = round r of the batch (its cells share no dof), CPB = the plan's
// W slots; consecutive rounds DO share dofs, so the update of y in round r waits (mbarrier, split
// arrive / wait like the brick kernel's) until every warp has finished round r-1's.  The batch's dofs
// are then touched by one SM within a few microseconds: x gathers hit L1 / L2 and the read-modify-write
// of y stays in L2, so DRAM sees what the brick kernel's staging moves -- without the shared-memory dof
// arrays (two CTAs per SM at P4, three at P7), without the staging / write-back phases that keep a CTA
// of that kernel waiting on memory for a third of its life, and with L1 nearly whole.  Batches of one
// (execution) colour share no dof; FIRST / LAST follow the order (colour, round).
template <typename T, int N, int SLOT, int CPB, int MINB, int GW, bool BRICK>
__global__ void __launch_bounds__(SLOT* CPB, MINB)
stiff_cell2_kernel(const Cell2Args<T> a, const DMat<T, N> Dm, int cell0, int ncl)
{
  constexpr int N2 = N * N, ND = N2 * N, NT = SLOT * CPB;
  using V2 = typename Vec2<T>::type;
  using L = LayoutStd<N, sizeof(T)>;
  static_assert(SLOT <= 32 ? (32 % SLOT == 0) : (SLOT % 32 == 0), "a slot is a fraction or a multiple of a warp");
  static_assert(SLOT <= 32 || CPB <= 15, "one named barrier per slot");
  static_assert(!BRICK || NT % 32 == 0, "whole warps");
  __shared__ __align__(16) T s_w[CPB][L::SLOT_ELEMS];
  __shared__ __align__(8) uint64_t s_rbar;
  constexpr bool RB = BRICK && NT > 32; // round barrier needed (one warp: program order suffices)
  if (RB && threadIdx.x == 0) mbar_init(&s_rbar, NT / 32); // one arrival per warp and round
  pdl_launch_dependents(); // the next colour may start gathering; it waits before touching y
  const int slot = threadIdx.x / SLOT, col = threadIdx.x % SLOT;
  const bool lane_ok = col < N2;
  const RoleOff ro = L::offsets(lane_ok ? col : 0);
  const int gcol = g_column<L, N>(ro, lane_ok ? col : 0, a.g_order);
  // colour-ordered: this slot's cells are a.cps consecutive entries of the colour's list;
  // brick-ordered: cell0 + blockIdx.x is the batch, its rounds are the iterations
  int first = 0, r0 = 0, niter = a.cps;
  if constexpr (BRICK)
  {
    const int b = cell0 + (int)blockIdx.x;
    r0 = a.uni_nr ? b * a.uni_nr : __ldg(a.round_off + b);
    niter = a.uni_nr ? a.uni_nr : __ldg(a.round_off + b + 1) - r0;
  }
  else first = ((int)blockIdx.x * CPB + slot) * a.cps;
  auto cell_at = [&](int i) -> int {
    if constexpr (BRICK) return i < niter ? __ldg(a.slot_cell + (int64_t)(r0 + i) * CPB + slot) : -1;
    else return (i < a.cps && first + i < ncl) ? __ldg(a.cells + cell0 + first + i) : -1;
  };
  if constexpr (RB) __syncthreads(); // the barrier is initialised before anyone arrives
  auto sync = [&]() {
    if constexpr (SLOT <= 32) __syncwarp();
    else SlotBarSync{slot + 1, SLOT}();
  };
  int cell = cell_at(0), cn = cell_at(1);
  WFX_DEV_ASSERT(cell < a.ncells && cn < a.ncells);
  uint32_t dof[N];
  T u[N];
  V2 g[GW][3];
#pragma unroll
  for (int k = 0; k < N; ++k)
    dof[k] = (lane_ok && cell >= 0) ? ld_once(a.tdmf + (int64_t)cell * ND + k * N2 + col) : BD_HOLE;
  if (lane_ok && cell >= 0) load_G<T, N, GW>(a.G6 + (int64_t)cell * (6 * ND), gcol, g);
  if constexpr ((6 * ND * sizeof(T)) % 16 == 0)
    if (col == 0 && cn >= 0) l2_prefetch_bulk(a.G6 + (int64_t)cn * (6 * ND), (uint32_t)(6 * ND * sizeof(T)));
#pragma unroll
  for (int k = 0; k < N; ++k)
  {
    WFX_DEV_ASSERT(dof[k] == BD_HOLE || (int64_t)(dof[k] & BD_MASK) < a.ndofs);
    u[k] = dof[k] != BD_HOLE ? __ldg(a.x + (dof[k] & BD_MASK)) : T(0);
  }
  bool waited = false;
  T* tiles = s_w[slot];
  PhaseTimer tm;
  tm.start(false);
  for (int it = 0; it < niter; ++it)
  {
    const bool active = lane_ok && cell >= 0;
    const int cnn = cell_at(it + 2);
    WFX_DEV_ASSERT(cnn < a.ncells);
    uint32_t dofn[N];
#pragma unroll
    for (int k = 0; k < N; ++k)
      dofn[k] = (lane_ok && cn >= 0) ? ld_once(a.tdmf + (int64_t)cn * ND + k * N2 + col) : BD_HOLE;
    if constexpr ((6 * ND * sizeof(T)) % 16 == 0)
      if (col == 0 && cnn >= 0) l2_prefetch_bulk(a.G6 + (int64_t)cnn * (6 * ND), (uint32_t)(6 * ND * sizeof(T)));
    const V2* gcur = active ? reinterpret_cast<const V2*>(a.G6 + (int64_t)cell * (6 * ND)) + gcol : nullptr;
    const V2* gnext = (lane_ok && cn >= 0) ? reinterpret_cast<const V2*>(a.G6 + (int64_t)cn * (6 * ND)) + gcol : nullptr;
    T f2[N], yv[N];
    if constexpr (SLOT <= 32) cell_part1<T, N, L, GW>(u, g, tiles, ro, Dm, a.coeff, active, WarpSync(), f2, tm, gcur, gnext);
    else cell_part1<T, N, L, GW>(u, g, tiles, ro, Dm, a.coeff, active, SlotBarSync{slot + 1, SLOT}, f2, tm, gcur, gnext);
    // u is consumed: its registers take the next cell's x values, in flight during part 2
#pragma unroll
    for (int k = 0; k < N; ++k)
    {
      WFX_DEV_ASSERT(dofn[k] == BD_HOLE || (int64_t)(dofn[k] & BD_MASK) < a.ndofs);
      u[k] = dofn[k] != BD_HOLE ? __ldg(a.x + (dofn[k] & BD_MASK)) : T(0);
    }
    // a slot that idles in this round has requested nothing inside the G multiply: load the next cell's
    // window now (batches of a brick plan leave slots empty in some rounds)
    if (lane_ok && cn >= 0 && !active) load_G<T, N, GW>(a.G6 + (int64_t)cn * (6 * ND), gcol, g);
    T yo[N], sc[N];
    auto request_y = [&]() {
      if (!waited)
      {
        pdl_wait(); // earlier colours have finished their writes to y
        waited = true;
      }
      if constexpr (RB)
        if (it > 0) mbar_wait(&s_rbar, (it - 1) & 1); // every warp has finished round it-1's update of y
#pragma unroll
      for (int k = 0; k < N; ++k)
      {
        const uint32_t e = dof[k];
        const bool ok = active; // (idle lanes hold BD_HOLE)
        yo[k] = (ok && (!(e & BD_FIRST) || a.beta)) ? __ldcg(a.y + (e & BD_MASK)) : T(0);
        sc[k] = (ok && (e & BD_LAST) && a.scale) ? ld_once(a.scale + (e & BD_MASK)) : T(1);
      }
    };
    if constexpr (SLOT <= 32) cell_part2<T, N, L>(f2, tiles, ro, Dm, active, WarpSync(), yv, tm);
    else cell_part2<T, N, L>(f2, tiles, ro, Dm, active, SlotBarSync{slot + 1, SLOT}, yv, tm);
    request_y();
    if (active)
    {
#pragma unroll
      for (int k = 0; k < N; ++k) a.y[dof[k] & BD_MASK] = (yo[k] + yv[k]) * sc[k];
    }
    sync(); // part 2's reads of the tiles precede the next cell's writes
    if constexpr (RB)
    {
      __syncwarp();
      if (it + 1 < niter && threadIdx.x % 32 == 0) mbar_arrive(&s_rbar); // (release: the warp's stores to y)
    }
    cell = cn;
    cn = cnn;
#pragma unroll
    for (int k = 0; k < N; ++k) dof[k] = dofn[k];
  }
  if (!waited) pdl_wait();
}

// ---- ensemble kernel: nv fields per pass over G and the dofmap -------------------------------
// Vectors are member-interleaved (entry (dof i, member m) at i*nv + m: DOLFINx's blocked layout with
// bs = nv).  Cells run in colour order as in stiff_cell2_kernel -- no dof arrays in shared memory,
// FIRST / LAST flags in the per-point dofmap -- one cell per slot.  The slot loads the cell's dof
// indices and its whole G (N planes, GW = N) into registers once and then runs the sum-factorised
// kernel once per member, so G and the dofmap stream from HBM once for all members while a dof's nv
// values are one contiguous span of nv*sizeof(T) bytes: the gather / update of member m + 1 hits the
// sectors member m brought into L1 / L2.  The next member's x values are gathered while the current
// member finishes part 2.  nv is a run-time value: one instantiation serves every nv.
template <typename T>
struct EnsArgs
{
  const int32_t* cells;  // cell ids sorted by colour
  const uint32_t* tdmf;  // [ncells][ND] k-major point order: global dof | BD_FIRST | BD_LAST
  const T* G6;
  const T* x;            // [ndofs][nv]
  T* y;                  // [ndofs][nv]
  const T* scale;        // [ndofs], nullable: applied on the LAST touch of a dof
  T coeff;
  int beta;    // 0: FIRST touch overwrites y; 1: accumulates into y
  int g_order; // column order of G6 (see g_column)
  int nv;
  int64_t ndofs, ncells;
};

template <typename T, int N, int SLOT, int CPB, int MINB>
__global__ void __launch_bounds__(SLOT* CPB, MINB)
stiff_ens_kernel(const EnsArgs<T> a, const DMat<T, N> Dm, int cell0, int ncl)
{
  constexpr int N2 = N * N, ND = N2 * N;
  using V2 = typename Vec2<T>::type;
  using L = LayoutStd<N, sizeof(T)>;
  static_assert(SLOT <= 32 ? (32 % SLOT == 0) : (SLOT % 32 == 0), "a slot is a fraction or a multiple of a warp");
  static_assert(SLOT <= 32 || CPB <= 15, "one named barrier per slot");
  __shared__ __align__(16) T s_w[CPB][L::SLOT_ELEMS];
  pdl_launch_dependents(); // the next colour may start gathering; it waits before touching y
  const int slot = threadIdx.x / SLOT, col = threadIdx.x % SLOT;
  const bool lane_ok = col < N2;
  const RoleOff ro = L::offsets(lane_ok ? col : 0);
  const int gcol = g_column<L, N>(ro, lane_ok ? col : 0, a.g_order);
  const int ci = (int)blockIdx.x * CPB + slot;
  const int cell = ci < ncl ? __ldg(a.cells + cell0 + ci) : -1;
  WFX_DEV_ASSERT(cell < a.ncells);
  const bool active = lane_ok && cell >= 0;
  const int nv = a.nv;
  auto sync = [&]() {
    if constexpr (SLOT <= 32) __syncwarp();
    else SlotBarSync{slot + 1, SLOT}();
  };
  uint32_t dof[N];
  T u[N];
  V2 g[N][3];
#pragma unroll
  for (int k = 0; k < N; ++k)
  {
    dof[k] = active ? ld_once(a.tdmf + (int64_t)cell * ND + k * N2 + col) : BD_HOLE;
    WFX_DEV_ASSERT(dof[k] == BD_HOLE || (int64_t)(dof[k] & BD_MASK) < a.ndofs);
  }
  if (active) load_G<T, N, N>(a.G6 + (int64_t)cell * (6 * ND), gcol, g);
  auto gather = [&](int m) {
#pragma unroll
    for (int k = 0; k < N; ++k)
      u[k] = dof[k] != BD_HOLE ? __ldg(a.x + (int64_t)(dof[k] & BD_MASK) * nv + m) : T(0);
  };
  gather(0);
  bool waited = false;
  T* tiles = s_w[slot];
  PhaseTimer tm;
  tm.start(false);
  for (int m = 0; m < nv; ++m)
  {
    T f2[N], yv[N];
    // G stays in its registers for every member (no window refill: gcur / gnext are null)
    if constexpr (SLOT <= 32) cell_part1<T, N, L, N>(u, g, tiles, ro, Dm, a.coeff, active, WarpSync(), f2, tm);
    else cell_part1<T, N, L, N>(u, g, tiles, ro, Dm, a.coeff, active, SlotBarSync{slot + 1, SLOT}, f2, tm);
    // u is consumed: its registers take the next member's x values, in flight during part 2
    if (m + 1 < nv) gather(m + 1);
    if constexpr (SLOT <= 32) cell_part2<T, N, L>(f2, tiles, ro, Dm, active, WarpSync(), yv, tm);
    else cell_part2<T, N, L>(f2, tiles, ro, Dm, active, SlotBarSync{slot + 1, SLOT}, yv, tm);
    if (!waited)
    {
      pdl_wait(); // earlier colours have finished their writes to y
      waited = true;
    }
    if (active)
    {
      T yo[N], sc[N];
#pragma unroll
      for (int k = 0; k < N; ++k)
      {
        const uint32_t e = dof[k];
        yo[k] = (!(e & BD_FIRST) || a.beta) ? __ldcg(a.y + (int64_t)(e & BD_MASK) * nv + m) : T(0);
        sc[k] = ((e & BD_LAST) && a.scale) ? __ldg(a.scale + (e & BD_MASK)) : T(1);
      }
#pragma unroll
      for (int k = 0; k < N; ++k) a.y[(int64_t)(dof[k] & BD_MASK) * nv + m] = (yo[k] + yv[k]) * sc[k];
    }
    sync(); // part 2's reads of the tiles precede the next member's writes
  }
  if (!waited) pdl_wait();
}

// ---- product kernel: one CTA per batch ------------------------------------------------
template <typename T>
struct BrickArgs
{
  const int64_t* dof_off;
  const uint32_t* bdofs;
  const int32_t* round_off;
  const int32_t* slot_cell;
  const uint16_t* ldm;
  const T* G6;
  const T* Gc;    // AFF kernels: one symmetric 3x3 (6 entries) per cell
  const T* x;
  T* y;
  const T* scale; // nullable: applied on the LAST touch of a dof
  T coeff;
  int beta;       // 0: FIRST touch overwrites y; 1: accumulates into y
  int nloc_pad;   // capacity of the shared dof arrays (even)
  int rounds_max; // capacity (rounds) of the shared local-dofmap staging area
  int pf_stride;  // CTAs resident on the GPU at once (for the cross-CTA L2 prefetch)
  const uint16_t* slot_base; // REG kernels: position of each slot's origin corner
  int Sx, Sy;                // REG kernels: strides of the brick lattice in the shared arrays
  int g_order;               // column order of G6 (see g_column)
  int uni_nloc, uni_nr;      // > 0: every batch has this many dof positions / rounds (no header loads)
  const int32_t* batch_ids;  // IDS kernels (mixed plans): batch of CTA i is batch_ids[batch0 + i]
  int64_t ndofs, ncells;     // vector length / cell count (checked builds verify every index against them)
  int nbatches;
  int wait_first;            // first launch of an apply: wait for everything earlier in the stream before reading x
};

// Shared memory of one CTA
//   generic:  xl[nloc_pad] | yl[nloc_pad] | tiles[W][L::SLOT_ELEMS] | sldm[rounds_max*W*NDP] (u16)
//             | scell[rounds_max*W] (i32) | two mbarriers (TMA copy of sldm, round barrier)
//   REG:      xl | yl | tiles | scell[rounds_max*W] (i32) | sbase[rounds_max*W] (u16) | mbarriers
// REG: every batch of the launch is a regular brick (wfx_plan): the positions of a cell's points
// in the shared arrays are base + ascpos(i)*Sx + ascpos(j)*Sy + ascpos(k), so no local dofmap is
// staged and all three roles read their input lines straight from xl (no tile round trip for u).
// At P4 fp64 the REG layout is 99.1 KB: two CTAs fit the 196 KB carve-out, which leaves 60 KB of
// L1 -- do not grow it (DESIGN.md 4.2, "L1 is part of the budget").
// AFF (with REG): every cell is affine -- G(q) = w_q A_cell, 6 scalars per cell from a.Gc; the
// per-point array G6 is never read (structured fast path, SURVEY 8f-2).
// IDS: the batch of CTA i is a.batch_ids[batch0 + i] (mixed plans).  A separate instantiation: with
// the indirection the batch index is a loaded value instead of a uniform expression of blockIdx, and
// everything derived from it leaves the uniform datapath (measured: +25 % at P2 fp32).
template <typename T, int N, int SLOT, int W, int MINB, bool REG, typename L, bool AFF = false, bool IDS = false>
__global__ void __launch_bounds__(SLOT* W, MINB)
stiff_brick_kernel(const BrickArgs<T> a, const DMat<T, N> Dm, int batch0)
{
  static_assert(!AFF || REG, "the affine path is built for regular bricks only");
  // U: batch dofs handled per thread in one pass of the staging / write-back loops; all their
  // loads are issued before the first is consumed (two dependent memory round trips per pass)
  constexpr int N2 = N * N, ND = N2 * N, NT = SLOT * W, NDP = ndp_of<N>();
  constexpr int U = 21;
  // planes of G held in registers (rotating window, see g_multiply).  fp32 has the registers for the
  // whole next cell and is faster with it (P4: 0.271 vs 0.307 ms); fp64 uses the per-degree window.
  constexpr int GW = sizeof(T) == 4 ? N : Cfg<N>::GW;
  using V2 = typename Vec2<T>::type;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* xl = reinterpret_cast<T*>(smem_raw);
  T* yl = xl + a.nloc_pad;
  T* work = yl + a.nloc_pad;
  // 16-byte aligned for the bulk copy below
  const size_t meta_off = ((size_t)(2 * a.nloc_pad + W * L::SLOT_ELEMS) * sizeof(T) + 15) & ~(size_t)15;
  // generic: sldm | scell | mbarrier.   REG: scell | sbase (u16)
  uint16_t* sldm = reinterpret_cast<uint16_t*>(smem_raw + meta_off);
  int32_t* scell = REG ? reinterpret_cast<int32_t*>(smem_raw + meta_off)
                       : reinterpret_cast<int32_t*>(sldm + (size_t)a.rounds_max * W * NDP);
  uint16_t* sbase = reinterpret_cast<uint16_t*>(scell + (size_t)a.rounds_max * W);
  uint64_t* bar = reinterpret_cast<uint64_t*>(
      smem_raw + ((meta_off + (size_t)a.rounds_max * W * (REG ? 6 : NDP * 2 + 4) + 7) & ~(size_t)7));
  // Round barrier, split into arrive / wait when a cell is one warp's business (SLOT <= 32): only
  // the accumulation into yl has to wait for the previous round, everything before it (reads of
  // xl, the contractions in the warp's own tiles) runs ahead, and the warps drift apart instead of
  // hitting the same pipe in lock step.
#ifndef WFX_NO_SPLIT_BARRIER
  constexpr bool SPLIT = SLOT <= 32 && (SLOT * W) % 32 == 0 && SLOT * W > 32;
#else
  constexpr bool SPLIT = false;
#endif
  uint64_t* rbar = bar + 1;
  if (SPLIT && threadIdx.x == 0) mbar_init(rbar, NT / 32); // one arrival per warp and round
  pdl_launch_dependents(); // the next colour may start staging; it waits before touching y
  // The first launch of an apply is a programmatic dependent launch too: its CTAs are placed while the
  // kernel in front of it drains, and wait here -- x may be that kernel's output (0.4543 -> 0.4517 ms)
  if (a.wait_first) pdl_wait();
  PhaseTimer tm;
  tm.start(threadIdx.x % 32 == 0);
  const int b = IDS ? __ldg(a.batch_ids + batch0 + blockIdx.x) : batch0 + (int)blockIdx.x;
  WFX_DEV_ASSERT(b >= 0 && b < a.nbatches);
  // batch header: arithmetic when the plan is uniform (saves a memory round trip), else loaded
  const int64_t d0 = a.uni_nloc ? (int64_t)b * a.uni_nloc : __ldg(a.dof_off + b);
  const int nloc = a.uni_nloc ? a.uni_nloc : (int)(__ldg(a.dof_off + b + 1) - d0);
  const int tid = threadIdx.x;
  const int slot = tid / SLOT, col = tid % SLOT;
  const bool lane_ok = col < N2;
  const RoleOff ro = L::offsets(lane_ok ? col : 0);
  const int gcol = g_column<L, N>(ro, lane_ok ? col : 0, a.g_order);
  const int r0 = a.uni_nr ? b * a.uni_nr : __ldg(a.round_off + b);
  const int nr = a.uni_nr ? a.uni_nr : __ldg(a.round_off + b + 1) - r0;
  WFX_DEV_ASSERT(nloc >= 0 && nloc <= a.nloc_pad && nr >= 0 && nr <= a.rounds_max);

  // the batch's local dofmap: one TMA bulk copy, waited for after the dofs are staged
  if constexpr (!REG)
    if (tid == 0 && nr > 0) bulk_copy_g2s(sldm, a.ldm + (int64_t)r0 * W * NDP, (uint32_t)(nr * W * NDP * 2), bar);
  // REG: offsets of this thread's three lines relative to the cell's base position
  const int P1 = N - 1;
  auto apos = [P1](int q) { return q == 0 ? 0 : (q == 1 ? P1 : q - 1); };
  const int offK = apos(ro.iK) * a.Sx + apos(ro.jK) * a.Sy; // role K: line over k (stride 1)
  const int offJ = apos(ro.iJ) * a.Sx + apos(ro.kJ);        // role J: line over j (stride Sy)
  const int offI = apos(ro.jI) * a.Sy + apos(ro.kI);        // role I: line over i (stride Sx)

  // Staging.  A warp issues in order, so a load followed by its use costs a full memory round
  // trip before anything else can be issued: ALL loads that depend only on the batch header (the
  // dof indices of the first pass, the slot tables, the first cells) are issued back to back
  // into registers first and consumed afterwards -- two round trips instead of six.
  V2 g[GW][3];
  uint32_t e[U];
#pragma unroll
  for (int q = 0; q < U; ++q) e[q] = tid + q * NT < nloc ? ld_once(a.bdofs + d0 + tid + q * NT) : BD_HOLE;
  const int nslots = nr * W;
  const int sc_v = tid < nslots ? __ldg(a.slot_cell + (int64_t)r0 * W + tid) : -1;
  uint16_t sb_v = 0;
  if constexpr (REG) sb_v = tid < nslots ? __ldg(a.slot_base + (int64_t)r0 * W + tid) : (uint16_t)0;
  const int c0 = nr > 0 ? __ldg(a.slot_cell + (int64_t)r0 * W + slot) : -1;
  int cpf[PF_DIST > 0 ? PF_DIST : 1];
#pragma unroll
  for (int q = 1; q <= PF_DIST; ++q) cpf[q - 1] = q < nr ? __ldg(a.slot_cell + (int64_t)(r0 + q) * W + slot) : -1;
  // The G of the first 1 + PF_DIST rounds goes to L2 by bulk prefetch (one request per cell): the
  // register loads issued later are then L2 hits and leave the SM's load queue quickly.
  if constexpr ((6 * ND * sizeof(T)) % 16 == 0 && !AFF)
    if (col == 0)
    {
      if (c0 >= 0) l2_prefetch_bulk(a.G6 + (int64_t)c0 * (6 * ND), (uint32_t)(6 * ND * sizeof(T)));
#pragma unroll
      for (int q = 1; q <= PF_DIST; ++q)
        if (cpf[q - 1] >= 0) l2_prefetch_bulk(a.G6 + (int64_t)cpf[q - 1] * (6 * ND), (uint32_t)(6 * ND * sizeof(T)));
    }
  if (tid < nslots)
  {
    scell[tid] = sc_v;
    if constexpr (REG) sbase[tid] = sb_v;
  }
  for (int v = tid + NT; v < nslots; v += NT)
  {
    scell[v] = __ldg(a.slot_cell + (int64_t)r0 * W + v);
    if constexpr (REG) sbase[v] = __ldg(a.slot_base + (int64_t)r0 * W + v);
  }
  // the batch's dofs: asynchronous gathers into xl (first pass from the indices loaded above)
#ifdef WFX_STAGE_REG
  // experiment: gather through registers with L2-only loads (no L1 lines held by the gathers)
  {
    T xv[U];
#pragma unroll
    for (int q = 0; q < U; ++q) xv[q] = e[q] != BD_HOLE ? __ldcg(a.x + (e[q] & BD_MASK)) : T(0);
#pragma unroll
    for (int q = 0; q < U; ++q)
    {
      if (e[q] != BD_HOLE) xl[tid + q * NT] = xv[q];
      if (tid + q * NT < nloc) yl[tid + q * NT] = T(0);
    }
  }
#else
#pragma unroll
  for (int q = 0; q < U; ++q)
  {
    WFX_DEV_ASSERT(e[q] == BD_HOLE || (int64_t)(e[q] & BD_MASK) < a.ndofs);
    if (e[q] != BD_HOLE) cp_async_scalar(xl + tid + q * NT, a.x + (e[q] & BD_MASK));
    if (tid + q * NT < nloc) yl[tid + q * NT] = T(0);
  }
#endif
  for (int base = tid + NT * U; base < nloc; base += NT * U)
  {
#pragma unroll
    for (int q = 0; q < U; ++q) e[q] = base + q * NT < nloc ? ld_once(a.bdofs + d0 + base + q * NT) : BD_HOLE;
#pragma unroll
    for (int q = 0; q < U; ++q)
    {
      WFX_DEV_ASSERT(e[q] == BD_HOLE || (int64_t)(e[q] & BD_MASK) < a.ndofs);
      if (e[q] != BD_HOLE) cp_async_scalar(xl + base + q * NT, a.x + (e[q] & BD_MASK));
      if (base + q * NT < nloc) yl[base + q * NT] = T(0);
    }
  }
  tm.mark(10);
  T ga[6], csk[N]; // AFF: the cell's matrix and coeff * w_i w_j w_k of this thread's column
  if constexpr (AFF)
  {
    T wi = 0, wj = 0; // (static indices into the parameter bank: no local copy of Dm)
#pragma unroll
    for (int q = 0; q < N; ++q)
    {
      if (q == ro.iK) wi = Dm.w[q];
      if (q == ro.jK) wj = Dm.w[q];
    }
    const T wij = a.coeff * wi * wj;
#pragma unroll
    for (int k = 0; k < N; ++k) csk[k] = wij * Dm.w[k];
#pragma unroll
    for (int q = 0; q < 6; ++q) ga[q] = c0 >= 0 ? __ldg(a.Gc + (int64_t)c0 * 6 + q) : T(0);
  }
  else if (lane_ok && c0 >= 0) load_G<T, N, GW>(a.G6 + (int64_t)c0 * (6 * ND), gcol, g);
  cp_async_wait_all();
  tm.mark(11);
  if constexpr (!REG)
    if (nr > 0) mbar_wait(bar, 0);
  __syncthreads();
  tm.mark(0);

  T* tiles = work + slot * L::SLOT_ELEMS;
  for (int r = 0; r < nr; ++r)
  {
    const int cell = scell[r * W + slot];
    WFX_DEV_ASSERT(cell < a.ncells);
    const bool active = lane_ok && cell >= 0;
    const int cn = r + 1 < nr ? scell[(r + 1) * W + slot] : -1;
    bool g_requested = false; // next cell's G already requested inside part 1
    int li[N];
    T u[N], yv[N], f2[N];
    // this thread's column of the next cell's G: requested plane by plane inside the G multiply
    const V2* gnext = (!AFF && cn >= 0) ? reinterpret_cast<const V2*>(a.G6 + (int64_t)cn * (6 * ND)) + gcol : nullptr;
    const V2* gcur = (!AFF && cell >= 0) ? reinterpret_cast<const V2*>(a.G6 + (int64_t)cell * (6 * ND)) + gcol : nullptr;
    g_requested = active;
    T gan[6]; // AFF: the next cell's matrix, requested a round ahead
    if constexpr (AFF)
    {
#pragma unroll
      for (int q = 0; q < 6; ++q) gan[q] = cn >= 0 ? __ldg(a.Gc + (int64_t)cn * 6 + q) : T(0);
    }
    if constexpr (REG)
    {
      const int base = active ? (int)sbase[r * W + slot] : 0;
      T lj[N], lI[N];
#pragma unroll
      for (int m = 0; m < N; ++m)
      {
        constexpr int P0 = N - 1;
        const int am = m == 0 ? 0 : (m == 1 ? P0 : m - 1); // ascpos(m), compile-time after unrolling
        li[m] = base + offK + am;
        WFX_DEV_ASSERT(!active || (li[m] >= 0 && li[m] < nloc && base + offJ + am * a.Sy < nloc && base + offI + am * a.Sx < nloc));
        u[m] = active ? xl[li[m]] : T(0);
        lj[m] = active ? xl[base + offJ + am * a.Sy] : T(0);
        lI[m] = active ? xl[base + offI + am * a.Sx] : T(0);
        yv[m] = 0;
      }
      if constexpr (AFF)
      {
        if constexpr (SLOT <= 32) cell_part1_reg_affine<T, N, L>(u, lj, lI, ga, csk, tiles, ro, Dm, active, WarpSync(), f2, tm);
        else cell_part1_reg_affine<T, N, L>(u, lj, lI, ga, csk, tiles, ro, Dm, active, BlockSync(), f2, tm);
#pragma unroll
        for (int q = 0; q < 6; ++q) ga[q] = gan[q];
      }
      else if constexpr (SLOT <= 32) cell_part1_reg<T, N, L, GW>(u, lj, lI, g, tiles, ro, Dm, a.coeff, active, WarpSync(), f2, tm, gcur, gnext);
      else cell_part1_reg<T, N, L, GW>(u, lj, lI, g, tiles, ro, Dm, a.coeff, active, BlockSync(), f2, tm, gcur, gnext);
    }
    else
    {
      const uint16_t* lrow = sldm + (r * W + slot) * NDP + ro.colK;
#pragma unroll
      for (int k = 0; k < N; ++k)
      {
        li[k] = active ? (int)lrow[k * N2] : 0;
        WFX_DEV_ASSERT(li[k] >= 0 && li[k] < nloc);
        u[k] = active ? xl[li[k]] : T(0);
        yv[k] = 0;
      }
      if constexpr (SLOT <= 32) cell_part1<T, N, L, GW>(u, g, tiles, ro, Dm, a.coeff, active, WarpSync(), f2, tm, gcur, gnext);
      else cell_part1<T, N, L, GW>(u, g, tiles, ro, Dm, a.coeff, active, BlockSync(), f2, tm, gcur, gnext);
    }
    // G of this cell is consumed: request the next cell's G into the same registers so
    // that the loads fly during part 2 and the next gather
    {
      if constexpr (!AFF)
        if (lane_ok && cn >= 0 && !g_requested) load_G<T, N, GW>(a.G6 + (int64_t)cn * (6 * ND), gcol, g);
      // keep the L2 prefetch PF_DIST rounds ahead of the register loads
      if constexpr ((6 * ND * sizeof(T)) % 16 == 0 && !AFF)
        if (col == 0 && r + 1 + PF_DIST < nr)
        {
          const int c2 = scell[(r + 1 + PF_DIST) * W + slot];
          if (c2 >= 0) l2_prefetch_bulk(a.G6 + (int64_t)c2 * (6 * ND), (uint32_t)(6 * ND * sizeof(T)));
        }
      // the write-back walks the batch's dof list again: keep it in L2 (it was read ~30 us ago)
      if (r == nr - 1 && tid == SLOT * (W > 1 ? 1 : 0))
      {
        const int64_t dn = d0 & ~(int64_t)3;
        l2_prefetch_bulk(a.bdofs + dn, (uint32_t)(((d0 + nloc + 3) & ~(int64_t)3) - dn) * 4u);
      }
      // In the last round, warm L2 for the CTA that will take this one's place on the SM
      // (blocks are dispatched in index order, a.pf_stride of them are resident): the first
      // cells' G, the batch's dof list and its local dofmap -- what that CTA waits for first.
      if (r == nr - 1 && col == 0 && (int)blockIdx.x + a.pf_stride < (int)gridDim.x)
      {
        const int bn = IDS ? __ldg(a.batch_ids + batch0 + blockIdx.x + a.pf_stride) : b + a.pf_stride;
        const int r0n = a.uni_nr ? bn * a.uni_nr : __ldg(a.round_off + bn);
        if constexpr ((6 * ND * sizeof(T)) % 16 == 0 && !AFF)
        {
          const int cq = __ldg(a.slot_cell + (int64_t)r0n * W + slot);
          if (cq >= 0) l2_prefetch_bulk(a.G6 + (int64_t)cq * (6 * ND), (uint32_t)(6 * ND * sizeof(T)));
        }
        if (slot == 0)
        {
          // (16-byte granules: the list is padded by 4 entries on the device)
          const int64_t dn0 = a.uni_nloc ? (int64_t)bn * a.uni_nloc : __ldg(a.dof_off + bn);
          const int64_t dn1 = a.uni_nloc ? dn0 + a.uni_nloc : __ldg(a.dof_off + bn + 1);
          const int64_t dn = dn0 & ~(int64_t)3;
          const uint32_t nbytes = (uint32_t)(((dn1 + 3) & ~(int64_t)3) - dn) * 4u;
          if (nbytes) l2_prefetch_bulk(a.bdofs + dn, nbytes);
          if constexpr (!REG)
          {
            const int nrn = a.uni_nr ? a.uni_nr : __ldg(a.round_off + bn + 1) - r0n;
            const uint32_t lbytes = (uint32_t)(nrn * W * NDP * 2);
            if (lbytes) l2_prefetch_bulk(a.ldm + (int64_t)r0n * W * NDP, lbytes);
          }
        }
      }
    }
    tm.mark(4);
    if constexpr (SLOT <= 32) cell_part2<T, N, L>(f2, tiles, ro, Dm, active, WarpSync(), yv, tm);
    else cell_part2<T, N, L>(f2, tiles, ro, Dm, active, BlockSync(), yv, tm);
    if constexpr (SPLIT)
      if (r > 0) mbar_wait(rbar, (r - 1) & 1); // every warp has finished round r-1's accumulation
    if (active)
    {
#pragma unroll
      for (int k = 0; k < N; ++k) yl[li[k]] += yv[k]; // cells of one round share no dof
    }
    tm.mark(6);
    if constexpr (SPLIT)
    {
      __syncwarp();
      if (r + 1 < nr && tid % 32 == 0) mbar_arrive(rbar);
    }
    else __syncthreads();
    tm.mark(7);
  }
  if constexpr (SPLIT) __syncthreads();
  // write-back: every batch dof exactly once.  Index loads first, then (after the earlier
  // colours have finished) all y / scale loads of the pass, then the stores.
  for (int base = tid; base < nloc; base += NT * U)
  {
    uint32_t e[U];
    T v[U], sc[U];
#pragma unroll
    for (int q = 0; q < U; ++q) e[q] = base + q * NT < nloc ? ld_once(a.bdofs + d0 + base + q * NT) : BD_HOLE;
    if (base == tid)
    {
      pdl_wait(); // earlier colours have finished their writes to y
      tm.mark(8);
    }
#pragma unroll
    for (int q = 0; q < U; ++q)
    {
      const bool ok = e[q] != BD_HOLE; // in range and a real dof (regular bricks have unused positions)
      const uint32_t dof = e[q] & BD_MASK;
      WFX_DEV_ASSERT(!ok || (int64_t)dof < a.ndofs);
      v[q] = (ok && (!(e[q] & BD_FIRST) || a.beta)) ? __ldcg(a.y + dof) : T(0);
      sc[q] = (ok && (e[q] & BD_LAST) && a.scale) ? ld_once(a.scale + dof) : T(1);
    }
#pragma unroll
    for (int q = 0; q < U; ++q)
      if (e[q] != BD_HOLE) a.y[e[q] & BD_MASK] = (v[q] + yl[base + q * NT]) * sc[q];
  }
  if (nloc <= tid) pdl_wait(); // threads without a batch dof still honour the dependency
  tm.mark(9);
  tm.flush(b * W + slot);
}

// ---- product kernel, single-launch form: one resident CTA walks many batches -----------------
// The multi-launch kernel above pays, around the rounds of every batch, two dependent memory round
// trips to stage the dofs and two more to write them back, with nothing of its own to overlap them.
// Here a CTA processes the batches  blockIdx.x, blockIdx.x + gridDim.x, ...  of the colour-sorted
// list in ONE cooperative launch per apply, and
//  * as soon as the last round of batch t is done the shared x array is dead: the dof list of the
//    CTA's next batch is loaded and its gather (cp.async) issued BEFORE batch t is written back, so
//    the gather's round trip runs under the write-back's;
//  * the G stream carries across batches (the last round requests the first cell of the next batch);
//  * colours are ordered inside the launch by per-batch completion flags: a batch adds to y only
//    after the batches that touched its dofs last (wfx_plan.h, dep_off / dep_ids) have written back
//    -- a point-to-point wait, not a barrier per colour (the round-1 experiment with per-colour
//    counters lost for that reason).  Dependencies point to earlier list positions only, every CTA
//    walks its positions in increasing order and all CTAs are co-resident (cooperative launch), so
//    the waits cannot deadlock.  Flags hold the apply's epoch and never need resetting.
// Regular bricks only (REG data path, LayoutStd); the affine form shares it (AFF).
struct PersistArgs
{
  const int32_t* dep_off;
  const int32_t* dep_ids;
  uint32_t* done;  // [nbatches] epoch of the last completed write-back
  uint32_t epoch;
  int nbatches;
  uint32_t stagger_ns; // start delay of the second half of the grid (the second CTA of every SM)
};

__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p)
{
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v)
{
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

template <typename T, int N, int SLOT, int W, int MINB, typename L, bool AFF>
__global__ void __launch_bounds__(SLOT* W, MINB)
stiff_brick_persist(const BrickArgs<T> a, const PersistArgs pa, const DMat<T, N> Dm)
{
  constexpr int N2 = N * N, ND = N2 * N, NT = SLOT * W;
  constexpr int U = 21;
  constexpr int GW = sizeof(T) == 4 ? N : Cfg<N>::GW;
  using V2 = typename Vec2<T>::type;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* xl = reinterpret_cast<T*>(smem_raw);
  T* yl = xl + a.nloc_pad;
  T* work = yl + a.nloc_pad;
  const size_t meta_off = ((size_t)(2 * a.nloc_pad + W * L::SLOT_ELEMS) * sizeof(T) + 15) & ~(size_t)15;
  int32_t* scell = reinterpret_cast<int32_t*>(smem_raw + meta_off);
  uint16_t* sbase = reinterpret_cast<uint16_t*>(scell + (size_t)a.rounds_max * W);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + ((meta_off + (size_t)a.rounds_max * W * 6 + 7) & ~(size_t)7));
#ifndef WFX_NO_SPLIT_BARRIER
  constexpr bool SPLIT = SLOT <= 32 && (SLOT * W) % 32 == 0 && SLOT * W > 32;
#else
  constexpr bool SPLIT = false;
#endif
  uint64_t* rbar = bar + 1;
  const int tid = threadIdx.x;
  const int slot = tid / SLOT, col = tid % SLOT;
  const bool lane_ok = col < N2;
  const RoleOff ro = L::offsets(lane_ok ? col : 0);
  const int gcol = g_column<L, N>(ro, lane_ok ? col : 0, a.g_order);
  const int P1 = N - 1;
  auto apos = [P1](int q) { return q == 0 ? 0 : (q == 1 ? P1 : q - 1); };
  const int offK = apos(ro.iK) * a.Sx + apos(ro.jK) * a.Sy;
  const int offJ = apos(ro.iJ) * a.Sx + apos(ro.kJ);
  const int offI = apos(ro.jI) * a.Sy + apos(ro.kI);
  T* tiles = work + slot * L::SLOT_ELEMS;
  PhaseTimer tm;
  tm.start(tid % 32 == 0);

  if (SPLIT && tid == 0) mbar_init(rbar, NT / 32);
  for (int l = tid; l < a.nloc_pad; l += NT) yl[l] = T(0); // kept zero by every write-back
  __syncthreads();

  // batch header: arithmetic when the plan is uniform, else loaded
  auto header = [&](int b, int64_t& d0, int& nloc, int& r0, int& nr) {
    d0 = a.uni_nloc ? (int64_t)b * a.uni_nloc : __ldg(a.dof_off + b);
    nloc = a.uni_nloc ? a.uni_nloc : (int)(__ldg(a.dof_off + b + 1) - d0);
    r0 = a.uni_nr ? b * a.uni_nr : __ldg(a.round_off + b);
    nr = a.uni_nr ? a.uni_nr : __ldg(a.round_off + b + 1) - r0;
    WFX_DEV_ASSERT(b >= 0 && b < pa.nbatches && nloc >= 0 && nloc <= a.nloc_pad && nr >= 0 && nr <= a.rounds_max);
  };
  // issue the staging of batch b: dof list -> registers -> asynchronous gather into xl; slot tables.
  // Completion is awaited with cp.async.wait_all + __syncthreads at the top of the batch loop.
  auto stage = [&](int b) {
    int64_t d0;
    int nloc, r0, nr;
    header(b, d0, nloc, r0, nr);
    uint32_t e[U];
#pragma unroll
    for (int q = 0; q < U; ++q) e[q] = tid + q * NT < nloc ? ld_once(a.bdofs + d0 + tid + q * NT) : BD_HOLE;
    const int nslots = nr * W;
    for (int v = tid; v < nslots; v += NT)
    {
      scell[v] = __ldg(a.slot_cell + (int64_t)r0 * W + v);
      sbase[v] = __ldg(a.slot_base + (int64_t)r0 * W + v);
    }
#pragma unroll
    for (int q = 0; q < U; ++q)
    {
      WFX_DEV_ASSERT(e[q] == BD_HOLE || (int64_t)(e[q] & BD_MASK) < a.ndofs);
      if (e[q] != BD_HOLE) cp_async_scalar(xl + tid + q * NT, a.x + (e[q] & BD_MASK));
    }
    for (int base = tid + NT * U; base < nloc; base += NT * U)
    {
#pragma unroll
      for (int q = 0; q < U; ++q) e[q] = base + q * NT < nloc ? ld_once(a.bdofs + d0 + base + q * NT) : BD_HOLE;
#pragma unroll
      for (int q = 0; q < U; ++q)
        if (e[q] != BD_HOLE) cp_async_scalar(xl + base + q * NT, a.x + (e[q] & BD_MASK));
    }
  };

  // The two CTAs of an SM must not walk their phases in lock step: one of them in its rounds while the
  // other stages / writes back is what two CTAs per SM are for.  Separate launches desynchronise by
  // themselves (a CTA starts when a slot frees); here the second half of the grid starts late.
  if (pa.stagger_ns && blockIdx.x >= (gridDim.x + 1) / 2)
  {
    for (uint32_t w = 0; w < pa.stagger_ns; w += 1000) __nanosleep(1000);
  }
  int t = blockIdx.x;
  V2 g[GW][3];
  T ga[6], csk[N];
  if constexpr (AFF)
  {
    T wi = 0, wj = 0;
#pragma unroll
    for (int q = 0; q < N; ++q)
    {
      if (q == ro.iK) wi = Dm.w[q];
      if (q == ro.jK) wj = Dm.w[q];
    }
    const T wij = a.coeff * wi * wj;
#pragma unroll
    for (int k = 0; k < N; ++k) csk[k] = wij * Dm.w[k];
  }
  if (t < pa.nbatches)
  {
    int64_t d0;
    int nloc, r0, nr;
    header(t, d0, nloc, r0, nr);
    const int c0 = nr > 0 ? __ldg(a.slot_cell + (int64_t)r0 * W + slot) : -1;
    if constexpr (AFF)
    {
#pragma unroll
      for (int q = 0; q < 6; ++q) ga[q] = c0 >= 0 ? __ldg(a.Gc + (int64_t)c0 * 6 + q) : T(0);
    }
    else
    {
      if constexpr ((6 * ND * sizeof(T)) % 16 == 0)
        if (col == 0 && c0 >= 0) l2_prefetch_bulk(a.G6 + (int64_t)c0 * (6 * ND), (uint32_t)(6 * ND * sizeof(T)));
      if (lane_ok && c0 >= 0) load_G<T, N, GW>(a.G6 + (int64_t)c0 * (6 * ND), gcol, g);
    }
    stage(t);
  }
  uint32_t phase_base = 0; // round-barrier phases completed so far (one per round but the last of a batch)
  for (; t < pa.nbatches; t += gridDim.x)
  {
    const int tn = t + gridDim.x;
    int64_t d0;
    int nloc, r0, nr;
    header(t, d0, nloc, r0, nr);
    // the first cells of this CTA's next batch (G stream and L2 prefetch carry across batches)
    int r0n = 0, nrn = 0;
    if (tn < pa.nbatches)
    {
      int64_t d0n;
      int nlocn;
      header(tn, d0n, nlocn, r0n, nrn);
    }
    const int cn_first = nrn > 0 ? __ldg(a.slot_cell + (int64_t)r0n * W + slot) : -1;
    const int cn_second = nrn > 1 ? __ldg(a.slot_cell + (int64_t)(r0n + 1) * W + slot) : -1;
    cp_async_wait_all();
    __syncthreads(); // the staged dofs and slot tables of batch t are visible
    tm.mark(0);
    // the dof lists this CTA walks next (write-back of t, staging of tn): keep them in L2
    if (tid == 0)
    {
      const int64_t dn = d0 & ~(int64_t)3;
      l2_prefetch_bulk(a.bdofs + dn, (uint32_t)(((d0 + nloc + 3) & ~(int64_t)3) - dn) * 4u);
    }
    if (tid == 32 && tn < pa.nbatches)
    {
      int64_t d0n;
      int nlocn, q0, q1;
      header(tn, d0n, nlocn, q0, q1);
      const int64_t dn = d0n & ~(int64_t)3;
      l2_prefetch_bulk(a.bdofs + dn, (uint32_t)(((d0n + nlocn + 3) & ~(int64_t)3) - dn) * 4u);
    }
    // G of the second round to L2 (the first round's was requested by the previous batch)
    if constexpr (!AFF && (6 * ND * sizeof(T)) % 16 == 0)
      if (col == 0 && nr > 1)
      {
        const int c1 = scell[W + slot];
        if (c1 >= 0) l2_prefetch_bulk(a.G6 + (int64_t)c1 * (6 * ND), (uint32_t)(6 * ND * sizeof(T)));
      }

    for (int r = 0; r < nr; ++r)
    {
      const int cell = scell[r * W + slot];
      WFX_DEV_ASSERT(cell < a.ncells);
      const bool active = lane_ok && cell >= 0;
      const int cn = r + 1 < nr ? scell[(r + 1) * W + slot] : cn_first;
      int li[N];
      T u[N], yv[N], f2[N];
      // (the G registers do not carry across the batch boundary: the write-back needs them; the next
      // batch's first cell is requested right after it and is an L2 hit by then)
      const V2* gnext = (!AFF && cn >= 0 && r + 1 < nr) ? reinterpret_cast<const V2*>(a.G6 + (int64_t)cn * (6 * ND)) + gcol : nullptr;
      const V2* gcur = (!AFF && cell >= 0) ? reinterpret_cast<const V2*>(a.G6 + (int64_t)cell * (6 * ND)) + gcol : nullptr;
      T gan[6];
      if constexpr (AFF)
      {
#pragma unroll
        for (int q = 0; q < 6; ++q) gan[q] = cn >= 0 ? __ldg(a.Gc + (int64_t)cn * 6 + q) : T(0);
      }
      const int base = active ? (int)sbase[r * W + slot] : 0;
      T lj[N], lI[N];
#pragma unroll
      for (int m = 0; m < N; ++m)
      {
        constexpr int P0 = N - 1;
        const int am = m == 0 ? 0 : (m == 1 ? P0 : m - 1);
        li[m] = base + offK + am;
        WFX_DEV_ASSERT(!active || (li[m] >= 0 && li[m] < nloc && base + offJ + am * a.Sy < nloc && base + offI + am * a.Sx < nloc));
        u[m] = active ? xl[li[m]] : T(0);
        lj[m] = active ? xl[base + offJ + am * a.Sy] : T(0);
        lI[m] = active ? xl[base + offI + am * a.Sx] : T(0);
        yv[m] = 0;
      }
      if constexpr (AFF)
      {
        if constexpr (SLOT <= 32) cell_part1_reg_affine<T, N, L>(u, lj, lI, ga, csk, tiles, ro, Dm, active, WarpSync(), f2, tm);
        else cell_part1_reg_affine<T, N, L>(u, lj, lI, ga, csk, tiles, ro, Dm, active, BlockSync(), f2, tm);
#pragma unroll
        for (int q = 0; q < 6; ++q) ga[q] = gan[q];
      }
      else if constexpr (SLOT <= 32) cell_part1_reg<T, N, L, GW>(u, lj, lI, g, tiles, ro, Dm, a.coeff, active, WarpSync(), f2, tm, gcur, gnext);
      else cell_part1_reg<T, N, L, GW>(u, lj, lI, g, tiles, ro, Dm, a.coeff, active, BlockSync(), f2, tm, gcur, gnext);
      if constexpr (!AFF)
      {
        // a slot that was idle in this round has requested nothing: load the next cell's window now
        if (lane_ok && cn >= 0 && !active && r + 1 < nr) load_G<T, N, GW>(a.G6 + (int64_t)cn * (6 * ND), gcol, g);
        // keep the L2 prefetch PF_DIST rounds ahead of the register loads, across the batch boundary
        if constexpr ((6 * ND * sizeof(T)) % 16 == 0)
          if (col == 0)
          {
            const int rr = r + 1 + PF_DIST;
            const int c2 = rr < nr ? scell[rr * W + slot] : (rr == nr ? cn_first : (rr == nr + 1 ? cn_second : -1));
            if (c2 >= 0) l2_prefetch_bulk(a.G6 + (int64_t)c2 * (6 * ND), (uint32_t)(6 * ND * sizeof(T)));
          }
      }
      tm.mark(4);
      if constexpr (SLOT <= 32) cell_part2<T, N, L>(f2, tiles, ro, Dm, active, WarpSync(), yv, tm);
      else cell_part2<T, N, L>(f2, tiles, ro, Dm, active, BlockSync(), yv, tm);
      if constexpr (SPLIT)
        if (r > 0) mbar_wait(rbar, (phase_base + r - 1) & 1);
      if (active)
      {
#pragma unroll
        for (int k = 0; k < N; ++k) yl[li[k]] += yv[k];
      }
      tm.mark(6);
      if constexpr (SPLIT)
      {
        __syncwarp();
        if (r + 1 < nr && tid % 32 == 0) mbar_arrive(rbar);
      }
      else __syncthreads();
      tm.mark(7);
    }
    if constexpr (SPLIT)
    {
      __syncthreads();
      if (nr > 0) phase_base += nr - 1;
    }
    // xl and the slot tables are dead.  Write this batch back and stage the next one in the same passes,
    // the write-back's loads in front: issued behind the ~5000 scattered gather requests of a staging
    // they would wait for those to drain (measured: the write-back took 4x longer that way).
    int64_t d0n = 0;
    int nlocn = 0;
    if (tn < pa.nbatches)
    {
      int q0, q1;
      header(tn, d0n, nlocn, q0, q1);
      for (int v = tid; v < q1 * W; v += NT)
      {
        scell[v] = __ldg(a.slot_cell + (int64_t)q0 * W + v);
        sbase[v] = __ldg(a.slot_base + (int64_t)q0 * W + v);
      }
    }
    tm.mark(10);
    // the batches that touched my dofs last have written back
    {
      const int q0 = __ldg(pa.dep_off + t), q1 = __ldg(pa.dep_off + t + 1);
      for (int q = q0 + tid; q < q1; q += NT)
      {
        const uint32_t* f = pa.done + __ldg(pa.dep_ids + q);
        while ((int32_t)(ld_acquire_gpu(f) - pa.epoch) < 0) __nanosleep(64);
      }
    }
    __syncthreads();
    tm.mark(8);
    constexpr int UW = WFX_PERSIST_UW;
    const int nmax = nloc > nlocn ? nloc : nlocn;
    for (int base = tid; base < nmax; base += NT * UW)
    {
      uint32_t e[UW], en[UW];
      T v[UW], sc[UW];
#pragma unroll
      for (int q = 0; q < UW; ++q)
      {
        e[q] = base + q * NT < nloc ? ld_once(a.bdofs + d0 + base + q * NT) : BD_HOLE;
        en[q] = base + q * NT < nlocn ? ld_once(a.bdofs + d0n + base + q * NT) : BD_HOLE;
      }
#pragma unroll
      for (int q = 0; q < UW; ++q)
      {
        const bool ok = e[q] != BD_HOLE;
        const uint32_t dof = e[q] & BD_MASK;
        WFX_DEV_ASSERT(!ok || (int64_t)dof < a.ndofs);
        // y is written by other SMs inside this launch: read it at L2
        v[q] = (ok && (!(e[q] & BD_FIRST) || a.beta)) ? __ldcg(a.y + dof) : T(0);
        sc[q] = (ok && (e[q] & BD_LAST) && a.scale) ? ld_once(a.scale + dof) : T(1);
      }
#pragma unroll
      for (int q = 0; q < UW; ++q)
      {
        WFX_DEV_ASSERT(en[q] == BD_HOLE || (int64_t)(en[q] & BD_MASK) < a.ndofs);
        if (en[q] != BD_HOLE) cp_async_scalar(xl + base + q * NT, a.x + (en[q] & BD_MASK));
      }
#pragma unroll
      for (int q = 0; q < UW; ++q)
        if (base + q * NT < nloc)
        {
          if (e[q] != BD_HOLE) a.y[e[q] & BD_MASK] = (v[q] + yl[base + q * NT]) * sc[q];
          yl[base + q * NT] = T(0);
        }
    }
    if constexpr (!AFF)
      if (lane_ok && cn_first >= 0) load_G<T, N, GW>(a.G6 + (int64_t)cn_first * (6 * ND), gcol, g);
    __syncthreads(); // every thread's stores to y precede the flag; yl is zero for the next batch
    tm.mark(9);
    if (tid == 0)
    {
      __threadfence();
      st_release_gpu(pa.done + t, pa.epoch);
    }
  }
  tm.flush(blockIdx.x * W + slot);
}

template <typename T>
__global__ void zero_entries_kernel(const int32_t* __restrict__ idx, int n, T* __restrict__ y)
{
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) y[idx[t]] = T(0);
}
// the same for member-interleaved vectors: all nv members of the listed dofs
template <typename T>
__global__ void zero_entries_ens_kernel(const int32_t* __restrict__ idx, int64_t n, int nv, T* __restrict__ y)
{
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < n) y[(int64_t)idx[t / nv] * nv + t % nv] = T(0);
}

// One-time in-place reordering of the columns of a degree-4 G6 (rows of 25 2-vectors, one warp
// per row): the row's column q moves to position c_p4d_colpos[q].
template <typename T>
__global__ void permute_g_columns_kernel(T* __restrict__ G6, int64_t nrows)
{
  constexpr int NC = 25;
  using V2 = typename Vec2<T>::type;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x % 32;
  if (row >= nrows) return;
  V2* r = reinterpret_cast<V2*>(G6) + row * NC;
  V2 v{};
  if (lane < NC) v = r[lane];
  __syncwarp();
  if (lane < NC) r[c_p4d_colpos[lane]] = v;
}

// per-degree launch configuration
//                          SLOT  W  brick edge  cells/block (simple)  min CTAs/SM (brick)
//                          preferred shared-memory carve-out in percent, fp64 / fp32 (0 = driver's choice)
//                          GW: planes of G held in registers (must not exceed N; N = whole cell one round ahead)
template <> struct Cfg<3> { static constexpr int SLOT = 16, W = 16, BX = 8, BY = 8, BZ = 8, CPB = 16, MINB = 2, CARVEOUT = 0, CARVEOUT32 = 0, GW = 3; };
template <> struct Cfg<4> { static constexpr int SLOT = 16, W = 8, BX = 4, BY = 4, BZ = 4, CPB = 16, MINB = 4, CARVEOUT = 0, CARVEOUT32 = 0, GW = 4; };
#ifndef WFX_P4_W
#define WFX_P4_W 8
#define WFX_P4_BE 4
#define WFX_P4_MINB 2
#endif
#ifndef WFX_P4_BZ
#define WFX_P4_BZ WFX_P4_BE
#endif
#ifndef WFX_P4_MINB32
#define WFX_P4_MINB32 WFX_P4_MINB
#endif
#ifndef WFX_P4_CARVE
#define WFX_P4_CARVE 0
#endif
#ifndef WFX_P4_GW
#define WFX_P4_GW 3
#endif
#ifndef WFX_P5_GW
#define WFX_P5_GW 3
#endif
#ifndef WFX_P6_GW
#define WFX_P6_GW 4
#endif
#ifndef WFX_P7_GW
#define WFX_P7_GW 4
#endif
#ifndef WFX_P6_MINB
#define WFX_P6_MINB 4 // five CTAs per SM cap the kernel at 168 registers and it spills ~100 B; four: 0 B, 0.606 -> 0.524 ms
#endif
#ifndef WFX_P7_BZ
#define WFX_P7_BZ 1 // 2x2x1 cells: 38 KB per CTA, four CTAs per SM at 227 registers (no spills): fp64 0.579 -> 0.540 ms
#endif
#ifndef WFX_P6_BZ
#define WFX_P6_BZ 2
#endif
#ifndef WFX_P7_MINB
#define WFX_P7_MINB 4
#endif
template <> struct Cfg<5> { static constexpr int SLOT = 32, W = WFX_P4_W, BX = WFX_P4_BE, BY = WFX_P4_BE, BZ = WFX_P4_BZ, CPB = 8, MINB = WFX_P4_MINB, CARVEOUT = WFX_P4_CARVE, CARVEOUT32 = 0, GW = WFX_P4_GW; };
#ifndef WFX_P5_W
#define WFX_P5_W 1
#endif
#ifndef WFX_P5_BX
#define WFX_P5_BX 2
#endif
#ifndef WFX_P5_MINB
#define WFX_P5_MINB 8
#endif
#ifndef WFX_P5_CARVE
#define WFX_P5_CARVE 58
#endif
#ifndef WFX_P5_SLOT
#define WFX_P5_SLOT 64
#endif
#ifndef WFX_P5_BY
#define WFX_P5_BY 2
#endif
#ifndef WFX_P5_BZ
#define WFX_P5_BZ 2
#endif
template <> struct Cfg<6> { static constexpr int SLOT = WFX_P5_SLOT, W = WFX_P5_W, BX = WFX_P5_BX, BY = WFX_P5_BY, BZ = WFX_P5_BZ, CPB = 4, MINB = WFX_P5_MINB, CARVEOUT = WFX_P5_CARVE, CARVEOUT32 = 0, GW = WFX_P5_GW; };
#ifndef WFX_P6_W
#define WFX_P6_W 1
#define WFX_P6_BX 2
#define WFX_P6_BY 2
#endif
#ifndef WFX_P7_W
#define WFX_P7_W 1
#define WFX_P7_BX 2
#define WFX_P7_BY 2
#endif
#ifndef WFX_P6_CARVE
#define WFX_P6_CARVE 72
#endif
template <> struct Cfg<7> { static constexpr int SLOT = 64, W = WFX_P6_W, BX = WFX_P6_BX, BY = WFX_P6_BY, BZ = WFX_P6_BZ, CPB = 4, MINB = WFX_P6_MINB, CARVEOUT = WFX_P6_CARVE, CARVEOUT32 = 58, GW = WFX_P6_GW; };
template <> struct Cfg<8> { static constexpr int SLOT = 64, W = WFX_P7_W, BX = WFX_P7_BX, BY = WFX_P7_BY, BZ = WFX_P7_BZ, CPB = 2, MINB = WFX_P7_MINB, CARVEOUT = 0, CARVEOUT32 = 0, GW = WFX_P7_GW; };

// per-degree configuration of the streamed-cell kernel (stiff_cell2_kernel): cells per CTA, min CTAs
// per SM, planes of G in the register window (fp64; fp32 holds a whole cell).  The slot width is
// Cfg<N>::SLOT.
#ifndef WFX_C2_P5_CPB
#define WFX_C2_P5_CPB 4
#endif
#ifndef WFX_C2_P5_MINB
#define WFX_C2_P5_MINB 2
#endif
#ifndef WFX_C2_P5_GW
#define WFX_C2_P5_GW 3
#endif
#ifndef WFX_C2_P6_CPB
#define WFX_C2_P6_CPB 4
#endif
#ifndef WFX_C2_P6_MINB
#define WFX_C2_P6_MINB 2
#endif
#ifndef WFX_C2_P6_GW
#define WFX_C2_P6_GW 2
#endif
#ifndef WFX_C2_P7_CPB
#define WFX_C2_P7_CPB 4
#endif
#ifndef WFX_C2_P7_MINB
#define WFX_C2_P7_MINB 2
#endif
#ifndef WFX_C2_P7_GW
#define WFX_C2_P7_GW 2
#endif
// smallest N = P + 1 for which WFX_STIFF_AUTO takes the streamed-cell kernel, per scalar type
#ifndef WFX_CELL2_MIN_N64
#define WFX_CELL2_MIN_N64 99
#endif
#ifndef WFX_CELL2_MIN_N32
#define WFX_CELL2_MIN_N32 8 // P7 fp32: 0.235 ms (colour order) / 0.294 (brick order) against 0.311 for the brick kernel
#endif
// fp32 at P6 / P7: planes of G in the register window and min CTAs per SM of the colour-ordered kernel.  With
// a two-plane window instead of the whole next cell the P7 kernel fits 80 registers without spills (three
// 256-thread CTAs, 24 warps per SM) or 64 with 80 B of spills (four CTAs, 32 warps); occupancy then hides the
// latency and walking one cell per slot is fastest: P7 fp32 0.276 (whole-cell window, two CTAs, two cells per
// slot) -> 0.242 (three CTAs) -> 0.235 ms (four CTAs) = 0.61 of the HBM peak.  P6 fp32 stays with the brick
// kernel (0.284 against 0.288 at best).
#ifndef WFX_C2_P7_GW32
#define WFX_C2_P7_GW32 2
#endif
#ifndef WFX_C2_P7_MINB32
#define WFX_C2_P7_MINB32 4
#endif
#ifndef WFX_C2_P6_GW32
#define WFX_C2_P6_GW32 7
#endif
#ifndef WFX_C2_P6_MINB32
#define WFX_C2_P6_MINB32 WFX_C2_P6_MINB
#endif
template <int N> struct Cfg2;
template <> struct Cfg2<3> { static constexpr int CPB = 16, MINB = 2, GW = 3; };
template <> struct Cfg2<4> { static constexpr int CPB = 16, MINB = 2, GW = 4; };
#ifndef WFX_C2_P4_GW
#define WFX_C2_P4_GW 3
#endif
#ifndef WFX_C2_P4_MINB
#define WFX_C2_P4_MINB 2
#endif
template <> struct Cfg2<5> { static constexpr int CPB = 8, MINB = WFX_C2_P4_MINB, GW = WFX_C2_P4_GW; };
template <> struct Cfg2<6> { static constexpr int CPB = WFX_C2_P5_CPB, MINB = WFX_C2_P5_MINB, GW = WFX_C2_P5_GW; };
template <> struct Cfg2<7> { static constexpr int CPB = WFX_C2_P6_CPB, MINB = WFX_C2_P6_MINB, GW = WFX_C2_P6_GW; };
template <> struct Cfg2<8> { static constexpr int CPB = WFX_C2_P7_CPB, MINB = WFX_C2_P7_MINB, GW = WFX_C2_P7_GW; };

// brick-ordered form of the streamed-cell kernel: slots per CTA (= cells per round) and brick shape.
// No shared-memory dof arrays, so the brick is free: it only has to offer W cells per colour class.
#ifndef WFX_C3_P4_W
#define WFX_C3_P4_W 8
#endif
#ifndef WFX_C3_P4_BX
#define WFX_C3_P4_BX 4
#endif
#ifndef WFX_C3_P4_BY
#define WFX_C3_P4_BY 4
#endif
#ifndef WFX_C3_P4_BZ
#define WFX_C3_P4_BZ 4
#endif
#ifndef WFX_C3_P4_MINB
#define WFX_C3_P4_MINB 2
#endif
#ifndef WFX_C3_HI_W
#define WFX_C3_HI_W 4
#endif
#ifndef WFX_C3_HI_BX
#define WFX_C3_HI_BX 4
#endif
#ifndef WFX_C3_HI_BY
#define WFX_C3_HI_BY 4
#endif
#ifndef WFX_C3_HI_BZ
#define WFX_C3_HI_BZ 2
#endif
#ifndef WFX_C3_HI_MINB
#define WFX_C3_HI_MINB 2
#endif

template <int N> struct Cfg3;
template <> struct Cfg3<3> { static constexpr int W = 16, BX = 8, BY = 8, BZ = 8, MINB = 2; };
template <> struct Cfg3<4> { static constexpr int W = 16, BX = 8, BY = 8, BZ = 4, MINB = 2; };
template <> struct Cfg3<5> { static constexpr int W = WFX_C3_P4_W, BX = WFX_C3_P4_BX, BY = WFX_C3_P4_BY, BZ = WFX_C3_P4_BZ, MINB = WFX_C3_P4_MINB; };
template <> struct Cfg3<6> { static constexpr int W = WFX_C3_HI_W, BX = WFX_C3_HI_BX, BY = WFX_C3_HI_BY, BZ = WFX_C3_HI_BZ, MINB = WFX_C3_HI_MINB; };
template <> struct Cfg3<7> { static constexpr int W = WFX_C3_HI_W, BX = WFX_C3_HI_BX, BY = WFX_C3_HI_BY, BZ = WFX_C3_HI_BZ, MINB = WFX_C3_HI_MINB; };
template <> struct Cfg3<8> { static constexpr int W = WFX_C3_HI_W, BX = WFX_C3_HI_BX, BY = WFX_C3_HI_BY, BZ = WFX_C3_HI_BZ, MINB = WFX_C3_HI_MINB; };

struct Cfg3Rt
{
  int W, BX, BY, BZ;
};
Cfg3Rt cfg3_rt(int N)
{
  switch (N)
  {
  case 3: return {Cfg3<3>::W, Cfg3<3>::BX, Cfg3<3>::BY, Cfg3<3>::BZ};
  case 4: return {Cfg3<4>::W, Cfg3<4>::BX, Cfg3<4>::BY, Cfg3<4>::BZ};
  case 5: return {Cfg3<5>::W, Cfg3<5>::BX, Cfg3<5>::BY, Cfg3<5>::BZ};
  case 6: return {Cfg3<6>::W, Cfg3<6>::BX, Cfg3<6>::BY, Cfg3<6>::BZ};
  case 7: return {Cfg3<7>::W, Cfg3<7>::BX, Cfg3<7>::BY, Cfg3<7>::BZ};
  case 8: return {Cfg3<8>::W, Cfg3<8>::BX, Cfg3<8>::BY, Cfg3<8>::BZ};
  }
  fail("stiffness: degree %d not supported (2..7)", N - 1);
}

// G6 of every cell with the tensor axes relabelled: kernel axis a' is mesh axis s[a'], so
// G'(a', b') = G(s[a'], s[b']) at the same physical point, stored in the kernel's plane / column order
// of the primed indices.  The operator is invariant under the relabelling (same 1-D matrices on all
// axes); what changes is which index runs along the lanes of the gather / update instructions.
template <typename T>
__global__ void permute_g_axes_kernel(int n, int64_t ncells, int s0, int s1, int s2, const T* __restrict__ in,
                                      T* __restrict__ out)
{
  using V2 = typename Vec2<T>::type;
  const int n2 = n * n;
  const int64_t gid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (gid >= ncells * n * n2) return;
  const int64_t c = gid / (n * n2);
  const int r = (int)(gid % (n * n2));
  const int kp = r / n2, colp = r % n2, ip = colp / n, jp = colp % n;
  int sidx[3];
  sidx[s0] = ip, sidx[s1] = jp, sidx[s2] = kp; // the point's indices on the mesh's own axes
  const V2* src = reinterpret_cast<const V2*>(in) + ((c * n + sidx[2]) * 3) * (int64_t)n2 + sidx[0] * n + sidx[1];
  const V2 p0 = src[0], p1 = src[n2], p2 = src[2 * n2];
  const T G[3][3] = {{p0.x, p0.y, p1.x}, {p0.y, p1.y, p2.x}, {p1.x, p2.x, p2.y}};
  V2* dst = reinterpret_cast<V2*>(out) + ((c * n + kp) * 3) * (int64_t)n2 + colp;
  V2 q;
  q.x = G[s0][s0], q.y = G[s0][s1];
  dst[0] = q;
  q.x = G[s0][s2], q.y = G[s1][s1];
  dst[n2] = q;
  q.x = G[s1][s2], q.y = G[s2][s2];
  dst[2 * n2] = q;
}

// min CTAs per SM of the brick kernels per scalar type (fp32 batches are half the size and the kernel
// needs fewer registers, so more CTAs can be resident)
template <typename T, int N>
constexpr int minb_of()
{
  if constexpr (sizeof(T) == 4 && N == 5) return WFX_P4_MINB32;
  else return Cfg<N>::MINB;
}

struct LaunchCfg
{
  int SLOT, W, BX, BY, BZ, CPB;
};
int slot_elems_rt(int N, int esz)
{
  switch (N)
  {
  case 3: return esz == 8 ? slot_elems<3, 8>() : slot_elems<3, 4>();
  case 4: return esz == 8 ? slot_elems<4, 8>() : slot_elems<4, 4>();
  case 5: return esz == 8 ? slot_elems<5, 8>() : slot_elems<5, 4>();
  case 6: return esz == 8 ? slot_elems<6, 8>() : slot_elems<6, 4>();
  case 7: return esz == 8 ? slot_elems<7, 8>() : slot_elems<7, 4>();
  case 8: return esz == 8 ? slot_elems<8, 8>() : slot_elems<8, 4>();
  }
  return 2 * N * N * N;
}
LaunchCfg launch_cfg(int N)
{
  switch (N)
  {
  case 3: return {Cfg<3>::SLOT, Cfg<3>::W, Cfg<3>::BX, Cfg<3>::BY, Cfg<3>::BZ, Cfg<3>::CPB};
  case 4: return {Cfg<4>::SLOT, Cfg<4>::W, Cfg<4>::BX, Cfg<4>::BY, Cfg<4>::BZ, Cfg<4>::CPB};
  case 5: return {Cfg<5>::SLOT, Cfg<5>::W, Cfg<5>::BX, Cfg<5>::BY, Cfg<5>::BZ, Cfg<5>::CPB};
  case 6: return {Cfg<6>::SLOT, Cfg<6>::W, Cfg<6>::BX, Cfg<6>::BY, Cfg<6>::BZ, Cfg<6>::CPB};
  case 7: return {Cfg<7>::SLOT, Cfg<7>::W, Cfg<7>::BX, Cfg<7>::BY, Cfg<7>::BZ, Cfg<7>::CPB};
  case 8: return {Cfg<8>::SLOT, Cfg<8>::W, Cfg<8>::BX, Cfg<8>::BY, Cfg<8>::BZ, Cfg<8>::CPB};
  }
  fail("stiffness: degree %d not supported (2..7)", N - 1);
}
} // namespace

struct wfx_stiffness
{
  wfx_ctx* ctx = nullptr;
  wfx_geom* geom = nullptr;
  int P = 0, N = 0, nd = 0, dtype = WFX_F64, mode = WFX_STIFF_AUTO;
  int64_t ncells = 0, ndofs = 0;
  double c0 = 0;
  bool use_pdl = true;
  double Dhost[WFX_MAXN * WFX_MAXN];
  double Whost[WFX_MAXN]; // 1-D GLL weights
  // simple path
  CellColourPlan cplan;
  DevBuf<int32_t> d_cells, d_tdm;
  // streamed-cell path (shares the colour plan): per-point dofmap with FIRST / LAST flags
  bool cell2 = false;
  bool cell2_brick = false; // cells in the order of a brick plan (one CTA per batch) instead of global colours
  int cell2_cps = 1; // colour order: cells a slot walks per launch
  int axis_perm[3] = {0, 1, 2}; // kernel axis a' is the mesh's tensor axis axis_perm[a'] (see detect_axis_perm)
  DevBuf<uint32_t> d_tdmf;
  DevBuf<unsigned char> d_G6perm; // private copy of G6 in the permuted axis order (empty: identity)
  // ensemble path (WFX_STIFF_ENSEMBLE): streamed cells in colour order over member-interleaved vectors.
  // An operator whose own path is the colour-ordered streamed kernel shares its plan and G; any other
  // builds its own plan (identity axes: G6 is read as stored, through its column order)
  bool ens = false;
  int64_t nshared = 0;
  CellColourPlan ens_plan; // cell ids live in d_ens_cells
  DevBuf<int32_t> d_ens_cells, d_ens_untouched;
  DevBuf<uint32_t> d_ens_tdmf;
  // brick path
  int ncolours = 0, nloc_pad = 0, W = 0, rounds_max = 0;
  int part_split = 0; // first execution colour of the interior part (distributed meshes)
  size_t smem_bytes = 0;
  std::vector<int32_t> colour_off;
  DevBuf<int64_t> d_dof_off;
  DevBuf<uint32_t> d_bdofs;
  DevBuf<int32_t> d_round_off, d_slot_cell, d_untouched;
  DevBuf<uint16_t> d_ldm;
  // regular-brick form (every batch a lattice brick): arithmetic positions, no staged dofmap
  int uni_nloc = 0, uni_nr = 0; // uniform plans: dof positions / rounds of every batch (else 0)
  int variant = 0; // 0 generic, 1 regular bricks, 2 regular bricks + the P4 fp64 conflict-free layout
  bool affine = false; // every cell affine and every batch regular: the kernels that never read G6
  // mixed plans: regular batches run the regular-brick kernel, the others the generic one (two
  // launches per colour); lists of batch ids per colour
  bool mixed = false;
  int n_regular = 0, nbatches = 0;
  std::vector<int32_t> reg_off, irr_off; // [ncolours+1] into d_reg_ids / d_irr_ids
  DevBuf<int32_t> d_reg_ids, d_irr_ids;
  // single-launch (persistent) form: write-back dependencies, completion flags, apply counter
  bool persistent = false;
  int persist_grid = 0;
  uint32_t epoch = 0;
  DevBuf<int32_t> d_dep_off, d_dep_ids;
  DevBuf<uint32_t> d_done;
  int Sx = 0, Sy = 0;
  size_t smem_bytes_reg = 0;
  DevBuf<uint16_t> d_slot_base;
  // host-call staging
  DevBuf<unsigned char> d_hx, d_hy;
  // batched host calls: two buffer pairs, three streams (H2D | apply | D2H)
  DevBuf<unsigned char> d_bx[2], d_by[2];
  cudaStream_t bs_h2d = nullptr, bs_cmp = nullptr, bs_d2h = nullptr;
  cudaEvent_t ev_x[2] = {nullptr, nullptr}, ev_y[2] = {nullptr, nullptr}, ev_fx[2] = {nullptr, nullptr},
              ev_fy[2] = {nullptr, nullptr};
  ~wfx_stiffness()
  {
    if (geom && d_G6perm.p)
    {
      auto& v = geom->g_copies;
      v.erase(std::remove(v.begin(), v.end(), (void*)d_G6perm.p), v.end());
    }
    for (cudaStream_t st : {bs_h2d, bs_cmp, bs_d2h})
      if (st) cudaStreamDestroy(st);
    for (int q = 0; q < 2; ++q)
      for (cudaEvent_t e : {ev_x[q], ev_y[q], ev_fx[q], ev_fy[q]})
        if (e) cudaEventDestroy(e);
  }
};

namespace
{
template <typename T, int N>
void launch_simple(wfx_stiffness* op, const T* x, T* y, cudaStream_t st)
{
  using C = Cfg<N>;
  DMat<T, N> Dm;
  for (int q = 0; q < N * N; ++q) Dm.d[q] = (T)op->Dhost[q];
  const T coeff = (T)(-1.0 * op->c0 * op->c0);
  for (int k = 0; k < op->cplan.ncolours; ++k)
  {
    const int beg = op->cplan.colour_off[k], ncl = op->cplan.colour_off[k + 1] - beg;
    if (ncl == 0) continue;
    const int grid = (ncl + C::CPB - 1) / C::CPB;
    stiff_cell_kernel<T, N, C::SLOT, C::CPB><<<grid, C::SLOT * C::CPB, 0, st>>>(
        op->d_cells.p + beg, ncl, op->d_tdm.p, (const T*)op->geom->G6, x, y, Dm, coeff,
        op->geom->g_colpos.empty() ? 0 : 1);
  }
  WFX_CUDA(cudaGetLastError());
}

template <int N>
struct Cell2Slot
{
  static constexpr int SLOT = Cfg<N>::SLOT <= 32 ? Cfg<N>::SLOT : 64;
};

template <typename T, int N>
void launch_cell2(wfx_stiffness* op, const T* x, const T* scale, T* y, int beta, int part, cudaStream_t st)
{
  using C2 = Cfg2<N>;
  using C3 = Cfg3<N>;
  using C = Cell2Slot<N>; // whole warps per slot
  constexpr int GW = sizeof(T) == 4 ? (N == 8 ? WFX_C2_P7_GW32 : (N == 7 ? WFX_C2_P6_GW32 : N)) : C2::GW;
  constexpr int MINB2 = sizeof(T) == 4 ? (N == 8 ? WFX_C2_P7_MINB32 : (N == 7 ? WFX_C2_P6_MINB32 : C2::MINB)) : C2::MINB;
  DMat<T, N> Dm;
  for (int q = 0; q < N * N; ++q) Dm.d[q] = (T)op->Dhost[q];
  for (int q = 0; q < N; ++q) Dm.w[q] = (T)op->Whost[q];
  Cell2Args<T> a;
  a.cells = op->d_cells.p;
  a.tdmf = op->d_tdmf.p;
  a.G6 = op->d_G6perm.n ? (const T*)op->d_G6perm.p : (const T*)op->geom->G6;
  a.x = x;
  a.y = y;
  a.scale = scale;
  a.coeff = (T)(-1.0 * op->c0 * op->c0);
  a.beta = beta;
  // the private copy was made from G6 in its natural column order: a column reorder of the geometry by
  // an operator created later leaves it as it is
  a.g_order = (op->d_G6perm.n || op->geom->g_colpos.empty()) ? 0 : 1;
  a.cps = op->cell2_cps;
  a.ndofs = op->ndofs;
  a.ncells = op->ncells;
  a.round_off = op->d_round_off.p;
  a.slot_cell = op->d_slot_cell.p;
  a.uni_nr = op->uni_nr;
  if (!beta && op->d_untouched.n && part != 1)
  {
    const int n = (int)op->d_untouched.n;
    zero_entries_kernel<T><<<(n + 255) / 256, 256, 0, st>>>(op->d_untouched.p, n, y);
  }
  // the first launch must see everything earlier in the stream (x may be fresh); later launches chain
  // by programmatic dependent launch.  The interior part continues the interface part (launch_brick).
  const bool iface_nonempty = op->cell2_brick && op->part_split > 0 && op->colour_off[op->part_split] > op->colour_off[0];
  bool first = !(part == 1 && iface_nonempty);
  auto launch = [&](auto kern, int threads, int grid, int i0, int i1) {
    if (grid == 0) return;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (op->use_pdl && !first) ? 1 : 0;
    WFX_CUDA(cudaLaunchKernelEx(&cfg, kern, a, Dm, i0, i1));
    first = false;
  };
  if (op->cell2_brick)
  {
    if (op->W != C3::W) fail("stiffness: plan built for %d slots, kernel has %d", op->W, C3::W);
    const int k0 = part == 1 ? op->part_split : 0;
    const int k1 = part == 0 ? op->part_split : op->ncolours;
    for (int k = k0; k < k1; ++k)
      launch(stiff_cell2_kernel<T, N, C::SLOT, C3::W, C3::MINB, GW, true>, C::SLOT * C3::W,
             op->colour_off[k + 1] - op->colour_off[k], op->colour_off[k], 0);
    return;
  }
  if (part >= 0) fail("stiffness: colour-ordered streamed cells have no interface / interior parts");
  for (int k = 0; k < op->cplan.ncolours; ++k)
  {
    const int beg = op->cplan.colour_off[k], ncl = op->cplan.colour_off[k + 1] - beg;
    const int per_cta = C2::CPB * op->cell2_cps;
    launch(stiff_cell2_kernel<T, N, C::SLOT, C2::CPB, MINB2, GW, false>, C::SLOT * C2::CPB,
           (ncl + per_cta - 1) / per_cta, beg, ncl);
  }
}

// ensemble kernel: the streamed kernel's slot width, 256 threads per CTA.  A slot holds its cell's whole G
// in registers; at fp64 from P5 up that does not fit 128 registers per thread next to the rest, so those
// instantiations take up to 255 (one 256-thread CTA per SM less)
template <typename T, int N>
struct CfgE
{
  static constexpr int SLOT = Cell2Slot<N>::SLOT;
  static constexpr int CPB = 256 / SLOT;
  static constexpr int MINB = (sizeof(T) == 8 && N >= 6) ? 1 : 2;
};

template <typename T, int N>
void launch_ens(wfx_stiffness* op, int nv, const T* x, const T* scale, T* y, int beta, cudaStream_t st)
{
  using C = CfgE<T, N>;
  DMat<T, N> Dm;
  for (int q = 0; q < N * N; ++q) Dm.d[q] = (T)op->Dhost[q];
  for (int q = 0; q < N; ++q) Dm.w[q] = (T)op->Whost[q];
  const bool share = op->cell2 && !op->cell2_brick; // the operator's own colour-ordered streamed plan
  const CellColourPlan& cp = share ? op->cplan : op->ens_plan;
  const DevBuf<int32_t>& untouched = share ? op->d_untouched : op->d_ens_untouched;
  EnsArgs<T> a;
  a.cells = share ? op->d_cells.p : op->d_ens_cells.p;
  a.tdmf = share ? op->d_tdmf.p : op->d_ens_tdmf.p;
  a.G6 = (share && op->d_G6perm.n) ? (const T*)op->d_G6perm.p : (const T*)op->geom->G6;
  a.x = x;
  a.y = y;
  a.scale = scale;
  a.coeff = (T)(-1.0 * op->c0 * op->c0);
  a.beta = beta;
  a.g_order = ((share && op->d_G6perm.n) || op->geom->g_colpos.empty()) ? 0 : 1; // (as launch_cell2)
  a.nv = nv;
  a.ndofs = op->ndofs;
  a.ncells = op->ncells;
  if (!beta && untouched.n)
  {
    const int64_t n = (int64_t)untouched.n * nv;
    zero_entries_ens_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(untouched.p, n, nv, y);
  }
  // the first launch sees everything earlier in the stream; later colours chain by programmatic
  // dependent launch and wait before their first access to y
  bool first = true;
  for (int k = 0; k < cp.ncolours; ++k)
  {
    const int beg = cp.colour_off[k], ncl = cp.colour_off[k + 1] - beg;
    if (ncl == 0) continue;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((ncl + C::CPB - 1) / C::CPB);
    cfg.blockDim = dim3(C::SLOT * C::CPB);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (op->use_pdl && !first) ? 1 : 0;
    WFX_CUDA(cudaLaunchKernelEx(&cfg, stiff_ens_kernel<T, N, C::SLOT, C::CPB, C::MINB>, a, Dm, beg, ncl));
    first = false;
  }
}

template <typename T, int N>
void launch_brick(wfx_stiffness* op, const T* x, const T* scale, T* y, int beta, int part, cudaStream_t st)
{
  using C = Cfg<N>;
  using KernPtr = void (*)(BrickArgs<T>, DMat<T, N>, int);
  const int variant = op->variant;
  const KernPtr kern_gen = stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), false, LayoutStd<N, sizeof(T)>>;
  KernPtr kern = kern_gen;
  size_t smem = op->smem_bytes;
  if (variant == 1) kern = stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), true, LayoutStd<N, sizeof(T)>>, smem = op->smem_bytes_reg;
  if (variant == 1 && op->affine) kern = stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), true, LayoutStd<N, sizeof(T)>, true>;
  if constexpr (N == 5 && sizeof(T) == 8)
    if (variant == 2) kern = stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), true, LayoutP4D>, smem = op->smem_bytes_reg;
  // experiment knob (DESIGN.md 4.2, "L1 is part of the budget"): extra dynamic shared memory per CTA
  static const size_t smem_pad = std::getenv("WFX_SMEM_PAD") ? (size_t)std::atoi(std::getenv("WFX_SMEM_PAD")) : 0;
  smem += smem_pad;
  DMat<T, N> Dm;
  for (int q = 0; q < N * N; ++q) Dm.d[q] = (T)op->Dhost[q];
  for (int q = 0; q < N; ++q) Dm.w[q] = (T)op->Whost[q];
  BrickArgs<T> a;
  a.dof_off = op->d_dof_off.p;
  a.bdofs = op->d_bdofs.p;
  a.round_off = op->d_round_off.p;
  a.slot_cell = op->d_slot_cell.p;
  a.ldm = op->d_ldm.p;
  a.G6 = (const T*)op->geom->G6;
  a.Gc = (const T*)op->geom->Gc;
  a.x = x;
  a.y = y;
  a.scale = scale;
  a.coeff = (T)(-1.0 * op->c0 * op->c0);
  a.beta = beta;
  a.nloc_pad = op->nloc_pad;
  a.rounds_max = op->rounds_max;
  a.pf_stride = minb_of<T, N>() * op->ctx->num_sms;
  a.slot_base = op->d_slot_base.p;
  a.Sx = op->Sx;
  a.Sy = op->Sy;
  a.g_order = op->geom->g_colpos.empty() ? 0 : 1;
  a.uni_nloc = op->uni_nloc;
  a.uni_nr = op->uni_nr;
  a.batch_ids = nullptr;
  a.ndofs = op->ndofs;
  a.ncells = op->ncells;
  a.nbatches = op->nbatches;
  if (!beta && op->d_untouched.n && part != 1)
  {
    const int n = (int)op->d_untouched.n;
    zero_entries_kernel<T><<<(n + 255) / 256, 256, 0, st>>>(op->d_untouched.p, n, y);
  }
  // The interior part continues the apply its interface part started (same x, earlier in this
  // stream): its first launch may overlap that part's tail like any later colour.  Only if the
  // interface part has batches at all -- otherwise the kernel in front of us is x's producer.
  // (A property of the plan, not of the call history: the operator keeps no per-apply state and
  // may be applied from several streams.)
  // single-launch form: whole applies of all-regular plans (not the interface / interior parts)
  if (op->persistent && part == -1 && variant == 1)
  {
    using PK = void (*)(BrickArgs<T>, PersistArgs, DMat<T, N>);
    PK pk = op->affine ? (PK)stiff_brick_persist<T, N, C::SLOT, C::W, minb_of<T, N>(), LayoutStd<N, sizeof(T)>, true>
                       : (PK)stiff_brick_persist<T, N, C::SLOT, C::W, minb_of<T, N>(), LayoutStd<N, sizeof(T)>, false>;
    if (op->persist_grid == 0)
    {
      int occ = 0;
      WFX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pk, C::SLOT * C::W, op->smem_bytes_reg));
      if (occ < 1) fail("stiffness: the single-launch kernel does not fit on an SM");
      op->persist_grid = std::min(op->nbatches, occ * op->ctx->num_sms);
      if (const char* e = std::getenv("WFX_PERSIST_GRID")) op->persist_grid = std::min(op->persist_grid, std::atoi(e));
      if (std::getenv("WFX_VERBOSE"))
        std::fprintf(stderr, "[wfx] single-launch kernel: %d CTAs per SM, grid %d, %d batches, %zu B shared memory\n", occ,
                     op->persist_grid, op->nbatches, op->smem_bytes_reg);
    }
    PersistArgs pa;
    pa.dep_off = op->d_dep_off.p;
    pa.dep_ids = op->d_dep_ids.p;
    pa.done = op->d_done.p;
    pa.epoch = ++op->epoch;
    pa.nbatches = op->nbatches;
    static const uint32_t stagger = std::getenv("WFX_STAGGER_NS") ? (uint32_t)std::atoi(std::getenv("WFX_STAGGER_NS")) : 15000u;
    pa.stagger_ns = stagger;
    void* args[] = {(void*)&a, (void*)&pa, (void*)&Dm};
    WFX_CUDA(cudaLaunchCooperativeKernel((void*)pk, dim3(op->persist_grid), dim3(C::SLOT * C::W), args,
                                         op->smem_bytes_reg, st));
    return;
  }
  const bool iface_nonempty = op->part_split > 0 && op->colour_off[op->part_split] > op->colour_off[0];
  bool first = !(part == 1 && iface_nonempty);
  // execution colours of the requested part: interface batches [0, part_split), interior the rest
  const int k0 = part == 1 ? op->part_split : 0;
  const int k1 = part == 0 ? op->part_split : op->ncolours;
  auto launch = [&](KernPtr kp, size_t smem_k, int beg, int nb, const int32_t* ids) {
    if (nb == 0) return;
    a.batch_ids = ids;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(nb);
    cfg.blockDim = dim3(C::SLOT * C::W);
    cfg.dynamicSmemBytes = smem_k;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    // the first colour must see everything earlier in the stream (x may have just been produced): it
    // waits at its start (wait_first); later colours overlap their staging with the previous colour's tail.
    a.wait_first = first ? 1 : 0;
    cfg.numAttrs = op->use_pdl ? 1 : 0;
    WFX_CUDA(cudaLaunchKernelEx(&cfg, kp, a, Dm, beg));
    first = false;
  };
  for (int k = k0; k < k1; ++k)
  {
    if (op->mixed)
    {
      // regular batches with the regular-brick kernel, the rest with the generic one; the two
      // launches of a colour touch disjoint dofs and chain like colours do
      launch(stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), true, LayoutStd<N, sizeof(T)>, false, true>, op->smem_bytes_reg + smem_pad,
             op->reg_off[k], op->reg_off[k + 1] - op->reg_off[k], op->d_reg_ids.p);
      launch(stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), false, LayoutStd<N, sizeof(T)>, false, true>, op->smem_bytes + smem_pad,
             op->irr_off[k], op->irr_off[k + 1] - op->irr_off[k], op->d_irr_ids.p);
    }
    else launch(kern, smem, op->colour_off[k], op->colour_off[k + 1] - op->colour_off[k], nullptr);
  }
}

// opt in to the large dynamic shared-memory carve-out once per operator (per device)
template <typename T, int N>
void configure_brick(wfx_stiffness* op)
{
  using C = Cfg<N>;
  const int optin = (int)op->ctx->smem_optin;
  WFX_CUDA(cudaFuncSetAttribute(stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), false, LayoutStd<N, sizeof(T)>>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  WFX_CUDA(cudaFuncSetAttribute(stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), true, LayoutStd<N, sizeof(T)>>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  WFX_CUDA(cudaFuncSetAttribute(stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), true, LayoutStd<N, sizeof(T)>, true>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  WFX_CUDA(cudaFuncSetAttribute(stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), true, LayoutStd<N, sizeof(T)>, false, true>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  WFX_CUDA(cudaFuncSetAttribute(stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), false, LayoutStd<N, sizeof(T)>, false, true>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  WFX_CUDA(cudaFuncSetAttribute(stiff_brick_persist<T, N, C::SLOT, C::W, minb_of<T, N>(), LayoutStd<N, sizeof(T)>, false>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  WFX_CUDA(cudaFuncSetAttribute(stiff_brick_persist<T, N, C::SLOT, C::W, minb_of<T, N>(), LayoutStd<N, sizeof(T)>, true>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  if constexpr (N == 5 && sizeof(T) == 8)
    WFX_CUDA(cudaFuncSetAttribute(stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), true, LayoutP4D>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
  // Shared-memory carve-out (percent of the SM's 228 KB): L1 is what is left, and L1 is the landing
  // buffer of the loads in flight (DESIGN.md 4.2).  Default: the driver's choice (max occupancy).
  int carve = sizeof(T) == 8 ? C::CARVEOUT : C::CARVEOUT32; // measured per degree (profiles/r1_degree_sweep.md)
  if (const char* e = std::getenv("WFX_CARVEOUT")) carve = std::atoi(e);
  if (carve > 0)
  {
    WFX_CUDA(cudaFuncSetAttribute(stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), false, LayoutStd<N, sizeof(T)>>,
                                  cudaFuncAttributePreferredSharedMemoryCarveout, carve));
    WFX_CUDA(cudaFuncSetAttribute(stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), true, LayoutStd<N, sizeof(T)>>,
                                  cudaFuncAttributePreferredSharedMemoryCarveout, carve));
    WFX_CUDA(cudaFuncSetAttribute(stiff_brick_kernel<T, N, C::SLOT, C::W, minb_of<T, N>(), true, LayoutStd<N, sizeof(T)>, true>,
                                  cudaFuncAttributePreferredSharedMemoryCarveout, carve));
    WFX_CUDA(cudaFuncSetAttribute(stiff_brick_persist<T, N, C::SLOT, C::W, minb_of<T, N>(), LayoutStd<N, sizeof(T)>, false>,
                                  cudaFuncAttributePreferredSharedMemoryCarveout, carve));
    WFX_CUDA(cudaFuncSetAttribute(stiff_brick_persist<T, N, C::SLOT, C::W, minb_of<T, N>(), LayoutStd<N, sizeof(T)>, true>,
                                  cudaFuncAttributePreferredSharedMemoryCarveout, carve));
  }
}
template <typename T>
void configure_any(wfx_stiffness* op)
{
  switch (op->N)
  {
  case 3: configure_brick<T, 3>(op); break;
  case 4: configure_brick<T, 4>(op); break;
  case 5: configure_brick<T, 5>(op); break;
  case 6: configure_brick<T, 6>(op); break;
  case 7: configure_brick<T, 7>(op); break;
  case 8: configure_brick<T, 8>(op); break;
  default: fail("stiffness: degree %d not supported", op->P);
  }
}

template <typename T>
void dispatch_apply(wfx_stiffness* op, const T* x, const T* scale, T* y, int beta, int part, cudaStream_t st)
{
  if (op->mode == WFX_STIFF_CELL_COLOUR)
  {
    if (scale) fail("stiffness: fused scaling needs the brick kernel");
    if (!beta) WFX_CUDA(cudaMemsetAsync(y, 0, (size_t)op->ndofs * sizeof(T), st));
    switch (op->N)
    {
    case 3: launch_simple<T, 3>(op, x, y, st); break;
    case 4: launch_simple<T, 4>(op, x, y, st); break;
    case 5: launch_simple<T, 5>(op, x, y, st); break;
    case 6: launch_simple<T, 6>(op, x, y, st); break;
    case 7: launch_simple<T, 7>(op, x, y, st); break;
    case 8: launch_simple<T, 8>(op, x, y, st); break;
    default: fail("stiffness: degree %d not supported", op->P);
    }
    return;
  }
  if (op->cell2)
  {
    switch (op->N)
    {
    case 3: launch_cell2<T, 3>(op, x, scale, y, beta, part, st); break;
    case 4: launch_cell2<T, 4>(op, x, scale, y, beta, part, st); break;
    case 5: launch_cell2<T, 5>(op, x, scale, y, beta, part, st); break;
    case 6: launch_cell2<T, 6>(op, x, scale, y, beta, part, st); break;
    case 7: launch_cell2<T, 7>(op, x, scale, y, beta, part, st); break;
    case 8: launch_cell2<T, 8>(op, x, scale, y, beta, part, st); break;
    default: fail("stiffness: degree %d not supported", op->P);
    }
    return;
  }
  switch (op->N)
  {
  case 3: launch_brick<T, 3>(op, x, scale, y, beta, part, st); break;
  case 4: launch_brick<T, 4>(op, x, scale, y, beta, part, st); break;
  case 5: launch_brick<T, 5>(op, x, scale, y, beta, part, st); break;
  case 6: launch_brick<T, 6>(op, x, scale, y, beta, part, st); break;
  case 7: launch_brick<T, 7>(op, x, scale, y, beta, part, st); break;
  case 8: launch_brick<T, 8>(op, x, scale, y, beta, part, st); break;
  default: fail("stiffness: degree %d not supported", op->P);
  }
}

void apply_any(wfx_stiffness* op, const void* x, const void* scale, void* y, int beta, void* stream, int part = -1)
{
  if (!op) fail("stiffness operator is NULL");
  if (!x || !y) fail("stiffness: NULL vector");
  if (x == y) fail("stiffness: x and y must not alias");
  if (op->ncells == 0)
  {
    if (!beta)
      WFX_CUDA(cudaMemsetAsync(y, 0, (size_t)op->ndofs * (op->dtype == WFX_F64 ? 8 : 4), (cudaStream_t)stream));
    return;
  }
  ScopedDevice sd(op->ctx->device);
  if (op->dtype == WFX_F64)
    dispatch_apply<double>(op, (const double*)x, (const double*)scale, (double*)y, beta, part, (cudaStream_t)stream);
  else
    dispatch_apply<float>(op, (const float*)x, (const float*)scale, (float*)y, beta, part, (cudaStream_t)stream);
}

template <typename T>
void dispatch_ens(wfx_stiffness* op, int nv, const T* x, const T* scale, T* y, int beta, cudaStream_t st)
{
  switch (op->N)
  {
  case 3: launch_ens<T, 3>(op, nv, x, scale, y, beta, st); break;
  case 4: launch_ens<T, 4>(op, nv, x, scale, y, beta, st); break;
  case 5: launch_ens<T, 5>(op, nv, x, scale, y, beta, st); break;
  case 6: launch_ens<T, 6>(op, nv, x, scale, y, beta, st); break;
  case 7: launch_ens<T, 7>(op, nv, x, scale, y, beta, st); break;
  case 8: launch_ens<T, 8>(op, nv, x, scale, y, beta, st); break;
  default: fail("stiffness: degree %d not supported", op->P);
  }
  WFX_CUDA(cudaGetLastError());
}
} // namespace

// shared with the mass / boundary operators
namespace wfx
{
int stiffness_dtype(const wfx_stiffness* op) { return op->dtype; }
bool stiffness_has_split(const wfx_stiffness* op) { return op->part_split > 0; }
// the single-launch form passes a per-apply epoch as a kernel argument: not replayable from a graph
bool stiffness_graph_safe(const wfx_stiffness* op) { return !op->persistent; }
bool stiffness_has_ensemble(const wfx_stiffness* op) { return op->ens; }
double stiffness_c0(const wfx_stiffness* op) { return op->c0; }
int64_t stiffness_nshared(const wfx_stiffness* op) { return op->nshared; }
const wfx_geom* stiffness_geom(const wfx_stiffness* op) { return op->geom; }

// tensor-ordered dofmap in the kernels' k-major point order
void build_tensor_dofmap(int P, int64_t ncells, int64_t ndofs, const int32_t* dofmap,
                         std::vector<int32_t>& tdm)
{
  const int n = P + 1, n2 = n * n, nd = n2 * n;
  std::vector<int32_t> perm(nd);
  tensor_perm(P, perm.data());
  tdm.resize((size_t)ncells * nd);
  int32_t* out = tdm.data();
  parallel_for(ncells, [&](int64_t c0, int64_t c1) {
    for (int64_t c = c0; c < c1; ++c)
      for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j)
          for (int k = 0; k < n; ++k)
          {
            const int32_t d = dofmap[c * nd + perm[(i * n + j) * n + k]];
            if (d < 0 || d >= ndofs) fail("dofmap entry %d out of range [0,%lld)", d, (long long)ndofs);
            out[c * nd + k * n2 + i * n + j] = d;
          }
  });
}
} // namespace wfx

#ifdef WFX_TIMING
// debug builds only: device buffer [nbatches*W][12] of int64 phase cycle counts
extern "C" int wfx_debug_set_timing_buffer(void* buf)
{
  WFX_API_BEGIN
  WFX_CUDA(cudaMemcpyToSymbol(g_wfx_timing, &buf, sizeof(buf)));
  WFX_API_END
}
#endif

extern "C" int wfx_stiffness_create(wfx_ctx* ctx, wfx_geom* geom, int64_t ndofs,
                                    const int32_t* dofmap_host, double c0, int flags,
                                    wfx_stiffness** out)
{
  return wfx_stiffness_create_partitioned(ctx, geom, ndofs, dofmap_host, c0, flags, 0, nullptr, out);
}

extern "C" int wfx_stiffness_create_partitioned(wfx_ctx* ctx, wfx_geom* geom, int64_t ndofs,
                                                const int32_t* dofmap_host, double c0, int flags,
                                                int64_t nshared, const int32_t* shared_dofs_host,
                                                wfx_stiffness** out)
{
  WFX_API_BEGIN
  if (!ctx || !geom || !out) fail("NULL argument");
  if (nshared < 0 || (nshared > 0 && !shared_dofs_host)) fail("bad shared dof list");
  std::vector<uint8_t> shared;
  if (nshared > 0)
  {
    shared.assign((size_t)ndofs, 0);
    for (int64_t i = 0; i < nshared; ++i)
    {
      if (shared_dofs_host[i] < 0 || shared_dofs_host[i] >= ndofs) fail("shared dof out of range");
      shared[shared_dofs_host[i]] = 1;
    }
  }
  if (geom->ctx != ctx) fail("geometry belongs to another context");
  if (ndofs < 0) fail("negative ndofs");
  if (ndofs >= (1ll << 31)) fail("more than 2^31 local dofs");
  bool split_parts = !(flags & WFX_STIFF_NO_SPLIT);
  const bool ensemble = (flags & WFX_STIFF_ENSEMBLE) != 0;
  flags &= ~(WFX_STIFF_NO_SPLIT | WFX_STIFF_ENSEMBLE);
  if (flags != WFX_STIFF_AUTO && flags != WFX_STIFF_CELL_COLOUR && flags != WFX_STIFF_CELL_STREAM)
    fail("unknown stiffness flags %d", flags);
  if (const char* e = std::getenv("WFX_SPLIT")) split_parts = std::atoi(e) != 0;
  ScopedDevice sd(ctx->device);
  auto op = std::make_unique<wfx_stiffness>();
  op->ctx = ctx;
  op->geom = geom;
  op->P = geom->P;
  op->N = geom->n;
  op->nd = geom->nq;
  op->dtype = geom->dtype;
  op->ncells = geom->ncells;
  op->ndofs = ndofs;
  op->c0 = c0;
  op->mode = flags;
  if (const char* e = std::getenv("WFX_PDL")) op->use_pdl = std::atoi(e) != 0;
  const LaunchCfg lc = launch_cfg(op->N);
  deriv_1d(op->P, op->Dhost, true);
  {
    double pts[WFX_MAXN];
    gll_points_weights(op->P, pts, op->Whost);
  }
  if (op->ncells > 0)
  {
    if (!dofmap_host) fail("dofmap is NULL");
    SetupTimer timer("stiffness_create");
    std::vector<int32_t> tdm;
    build_tensor_dofmap(op->P, op->ncells, ndofs, dofmap_host, tdm);
    timer.lap("tensor dofmap");
    // Streamed-cell kernel: on request, or by degree where it measured faster than the brick kernel
    // (profiles/r2_degree_sweep.md); whole-mesh applies only (no interface / interior parts) and not
    // on all-affine meshes, which have their own brick kernels.
    bool cell2 = flags == WFX_STIFF_CELL_STREAM;
    if (flags == WFX_STIFF_AUTO && geom->n_affine != op->ncells)
      cell2 = op->N >= (op->dtype == WFX_F64 ? WFX_CELL2_MIN_N64 : WFX_CELL2_MIN_N32);
    if (const char* e = std::getenv("WFX_CELL2"))
      if (flags == WFX_STIFF_AUTO) cell2 = std::atoi(e) != 0 && geom->n_affine != op->ncells;
    if (flags == WFX_STIFF_CELL_COLOUR)
    {
      build_cell_colour_plan(op->nd, op->ncells, ndofs, tdm.data(), op->cplan);
      op->d_cells.upload(op->cplan.cells);
      op->d_tdm.upload(tdm);
    }
    else if (cell2)
    {
      if (ndofs > (int64_t)BD_MASK) fail("stiffness: more than 2^30 local dofs");
      const int nd = op->nd, n = op->N, n2 = n * n;
      // order of the cells: batches of a brick plan (default) or global cell colours
      // (measured, profiles/r2_kernel_experiments.md: global colours are the faster order wherever the
      // streamed kernel wins at all; partitioned meshes need the batches for their interface part)
      op->cell2_brick = flags == WFX_STIFF_CELL_STREAM || nshared > 0;
      if (const char* e = std::getenv("WFX_STREAM_ORDER")) op->cell2_brick = std::strcmp(e, "colour") != 0;
      if (nshared > 0 && !op->cell2_brick) fail("stiffness: colour-ordered streamed cells do not take partitioned meshes");
      const Cfg3Rt c3 = cfg3_rt(op->N);
      bool relabel = geom->g_colpos.empty(); // (a G with reordered columns keeps the mesh's axes)
      if (const char* e = std::getenv("WFX_AXIS_PERM")) relabel = relabel && std::atoi(e) != 0;
      StreamPlan sp;
      build_stream_plan(op->P, op->ncells, ndofs, tdm.data(), geom->centroid.empty() ? nullptr : geom->centroid.data(),
                        geom->cell_ijk.empty() ? nullptr : geom->cell_ijk.data(), op->cell2_brick,
                        BrickShape(c3.BX, c3.BY, c3.BZ), c3.W, shared.empty() ? nullptr : shared.data(), split_parts,
                        relabel, sp);
      timer.lap("stream plan");
      if (std::getenv("WFX_VERIFY_PLAN")) verify_stream_plan(sp, tdm.data(), shared.empty() ? nullptr : shared.data());
      if (op->cell2_brick)
      {
        op->ncolours = sp.ncolours;
        op->part_split = sp.part_split;
        op->colour_off = sp.colour_off;
        op->W = sp.W;
        op->nbatches = sp.nbatches;
        op->rounds_max = sp.rounds_max;
        op->uni_nr = sp.uni_nr;
        op->d_round_off.upload(sp.round_off);
        op->d_slot_cell.upload(sp.slot_cell);
      }
      else
      {
        op->cplan.ncolours = sp.ncolours;
        op->cplan.colour_off = sp.colour_off;
        op->d_cells.upload(sp.cells);
        if (const char* e = std::getenv("WFX_CELL2_CPS")) op->cell2_cps = std::max(1, std::atoi(e));
      }
      for (int q = 0; q < 3; ++q) op->axis_perm[q] = sp.axis_perm[q];
      const int s0 = op->axis_perm[0], s1 = op->axis_perm[1], s2 = op->axis_perm[2];
      op->d_tdmf.upload(sp.tdmf);
      if (!sp.untouched.empty()) op->d_untouched.upload(sp.untouched);
      if (s0 != 0 || s1 != 1)
      {
        const size_t esz = op->dtype == WFX_F64 ? 8 : 4;
        op->d_G6perm.alloc((size_t)op->ncells * nd * 6 * esz);
        geom->g_copies.push_back(op->d_G6perm.p); // scaled with G6 from now on (wfx_geometry_scale_cells)
        const int64_t npts = op->ncells * nd;
        const unsigned grid = (unsigned)((npts + 255) / 256);
        if (op->dtype == WFX_F64)
          permute_g_axes_kernel<double><<<grid, 256>>>(n, op->ncells, s0, s1, s2, (const double*)geom->G6, (double*)op->d_G6perm.p);
        else
          permute_g_axes_kernel<float><<<grid, 256>>>(n, op->ncells, s0, s1, s2, (const float*)geom->G6, (float*)op->d_G6perm.p);
        WFX_CUDA(cudaGetLastError());
        WFX_CUDA(cudaDeviceSynchronize());
      }
      op->cell2 = true;
      timer.lap("flags + uploads");
    }
    else
    {
      const size_t esz = op->dtype == WFX_F64 ? 8 : 4;
      // two [N][N][N] tiles per cell slot + the staged local dofmap / cell list of a batch;
      // the latter depends on the plan (rounds per batch), so budget for the regular case
      // (brick_edge^3 cells, 8 colours) first and verify after planning
      const int ndp = (op->nd + 7) & ~7;
      auto meta_bytes = [&](int rounds) { return (size_t)rounds * lc.W * (ndp * 2 + 4); };
      const int rounds_guess = std::max(8, (lc.BX * lc.BY * lc.BZ + lc.W - 1) / lc.W);
      const size_t tiles_bytes = (size_t)lc.W * slot_elems_rt(op->N, (int)esz) * esz;
      const size_t work = tiles_bytes + meta_bytes(rounds_guess) + 32;
      const size_t avail = ctx->smem_optin > work + 1024 ? ctx->smem_optin - work - 1024 : 0;
      int nloc_cap = (int)std::min<size_t>(avail / (2 * esz), 65535);
      if (const char* e = std::getenv("WFX_NLOC_CAP")) nloc_cap = std::min(nloc_cap, std::atoi(e));
      BrickShape be(lc.BX, lc.BY, lc.BZ);
      if (const char* e = std::getenv("WFX_BRICK_EDGE")) be = BrickShape(std::max(1, std::atoi(e)));
      BrickPlan bp;
      build_brick_plan(op->P, op->ncells, ndofs, tdm.data(),
                       geom->centroid.empty() ? nullptr : geom->centroid.data(), be, lc.W, nloc_cap, bp,
                       shared.empty() ? nullptr : shared.data(), (int)esz, true,
                       geom->cell_ijk.empty() ? nullptr : geom->cell_ijk.data(), split_parts);
      timer.lap("brick plan");
      op->ncolours = bp.ncolours;
      op->part_split = bp.part_split;
      op->colour_off = bp.colour_off;
      op->W = bp.W;
      op->nloc_pad = (bp.nloc_max + 1) & ~1;
      op->rounds_max = bp.rounds_max;
      op->smem_bytes = (((size_t)op->nloc_pad * 2 * esz + tiles_bytes + 15) & ~(size_t)15)
                       + meta_bytes(bp.rounds_max) + 32; // + mbarriers
      if (op->smem_bytes > ctx->smem_optin) fail("stiffness: batch needs %zu B shared memory", op->smem_bytes);
      op->d_dof_off.upload(bp.dof_off);
      {
        bool un = bp.nbatches > 0, ur = bp.nbatches > 0;
        for (int b = 0; b < bp.nbatches; ++b)
        {
          un = un && bp.dof_off[b + 1] - bp.dof_off[b] == bp.dof_off[1];
          ur = ur && bp.round_off[b + 1] - bp.round_off[b] == bp.round_off[1];
        }
        if (std::getenv("WFX_NO_UNIFORM")) un = ur = false;
        op->uni_nloc = un ? (int)bp.dof_off[1] : 0;
        op->uni_nr = ur ? bp.round_off[1] : 0;
      }
      bp.bdofs.resize(bp.bdofs.size() + 4, BD_HOLE); // slack for the 16-byte granules of the L2 prefetches
      op->d_bdofs.upload(bp.bdofs);
      op->d_round_off.upload(bp.round_off);
      op->d_slot_cell.upload(bp.slot_cell);
      op->d_ldm.upload(bp.ldm);
      op->d_slot_base.upload(bp.slot_base);
      op->Sx = bp.Sx;
      op->Sy = bp.Sy;
      bool regular = bp.nbatches > 0 && bp.n_regular == bp.nbatches;
      if (const char* e = std::getenv("WFX_REGULAR")) regular = regular && std::atoi(e) != 0;
      size_t tiles_reg = tiles_bytes;
      op->variant = regular ? 1 : 0;
      if (regular && op->N == 5 && esz == 8 && bp.Sx % 16 == LayoutP4D::SX_MOD && bp.Sy % 16 == LayoutP4D::SY_MOD)
      {
        op->variant = 2;
        tiles_reg = (size_t)lc.W * LayoutP4D::SLOT_ELEMS * esz;
      }
      op->smem_bytes_reg = (((size_t)op->nloc_pad * 2 * esz + tiles_reg + 15) & ~(size_t)15)
                           + (size_t)bp.rounds_max * lc.W * 6 + 32;
      if (op->variant && op->smem_bytes_reg > ctx->smem_optin) op->variant = 0;
      op->n_regular = bp.n_regular;
      op->nbatches = bp.nbatches;
      // mixed plan: most batches are lattice bricks, some (unstructured patches, batches split for
      // capacity) are not -- run each kind with its own kernel instead of dropping everything to
      // the generic one
      {
        bool mixed = op->variant == 0 && bp.n_regular > 0 && 2 * bp.n_regular >= bp.nbatches
                     && op->smem_bytes_reg <= ctx->smem_optin && bp.batch_regular.size() == (size_t)bp.nbatches;
        if (const char* e = std::getenv("WFX_MIXED")) mixed = mixed && std::atoi(e) != 0;
        if (const char* e = std::getenv("WFX_REGULAR")) mixed = mixed && std::atoi(e) != 0;
        if (mixed)
        {
          std::vector<int32_t> reg_ids, irr_ids;
          op->reg_off.assign(1, 0);
          op->irr_off.assign(1, 0);
          for (int k = 0; k < bp.ncolours; ++k)
          {
            for (int b = bp.colour_off[k]; b < bp.colour_off[k + 1]; ++b)
              (bp.batch_regular[b] ? reg_ids : irr_ids).push_back(b);
            op->reg_off.push_back((int32_t)reg_ids.size());
            op->irr_off.push_back((int32_t)irr_ids.size());
          }
          // slack: the cross-CTA prefetch reads the id pf_stride entries ahead (guarded by gridDim)
          op->d_reg_ids.upload(reg_ids);
          op->d_irr_ids.upload(irr_ids);
          op->mixed = true;
        }
      }
      // single-launch form (all-regular plans): dependencies and completion flags
      op->d_dep_off.upload(bp.dep_off);
      op->d_dep_ids.upload(bp.dep_ids);
      op->d_done.alloc((size_t)std::max(1, bp.nbatches));
      WFX_CUDA(cudaMemset(op->d_done.p, 0, op->d_done.n * sizeof(uint32_t)));
      {
        int coop = 0;
        WFX_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device));
        op->persistent = op->variant == 1 && coop != 0 && WFX_PERSISTENT_DEFAULT;
        if (const char* e = std::getenv("WFX_PERSISTENT")) op->persistent = op->variant == 1 && coop != 0 && std::atoi(e) != 0;
      }
      // structured fast path: every cell affine and every batch a lattice brick
      op->affine = op->variant == 1 && geom->n_affine == op->ncells;
      if (const char* e = std::getenv("WFX_AFFINE")) op->affine = op->affine && std::atoi(e) != 0;
      // variant 2 reads G in the lane order of its role K: reorder the geometry's columns once
      // (in place; every other consumer honours geom->g_colpos)
      if (op->variant == 2 && geom->g_colpos.empty())
      {
        const int64_t nrows = op->ncells * op->N * 3;
        permute_g_columns_kernel<double><<<(unsigned)((nrows + 7) / 8), 256>>>((double*)geom->G6, nrows);
        WFX_CUDA(cudaGetLastError());
        WFX_CUDA(cudaDeviceSynchronize());
        geom->g_colpos.assign(h_p4d_colpos, h_p4d_colpos + 25);
      }
      if (!bp.untouched.empty()) op->d_untouched.upload(bp.untouched);
      if (op->dtype == WFX_F64) configure_any<double>(op.get());
      else configure_any<float>(op.get());
      timer.lap("uploads + configure");
    }
    // ensemble path: single-rank operators only (a blocked ghost exchange does not exist); it reuses the
    // operator's colour-ordered streamed plan when there is one
    if (ensemble && nshared == 0 && !(op->cell2 && !op->cell2_brick))
    {
      StreamPlan sp;
      build_stream_plan(op->P, op->ncells, ndofs, tdm.data(), nullptr, nullptr, false, BrickShape(1), 1, nullptr,
                        false, false, sp);
      timer.lap("ensemble plan");
      if (std::getenv("WFX_VERIFY_PLAN")) verify_stream_plan(sp, tdm.data());
      op->ens_plan.ncolours = sp.ncolours;
      op->ens_plan.colour_off = sp.colour_off;
      op->d_ens_cells.upload(sp.cells);
      op->d_ens_tdmf.upload(sp.tdmf);
      if (!sp.untouched.empty()) op->d_ens_untouched.upload(sp.untouched);
    }
  }
  op->nshared = nshared;
  op->ens = ensemble && nshared == 0;
  *out = op.release();
  WFX_API_END
}

extern "C" int wfx_stiffness_apply(wfx_stiffness* op, const void* x, void* y, int beta, void* stream)
{
  WFX_API_BEGIN
  apply_any(op, x, nullptr, y, beta, stream);
  WFX_API_END
}

extern "C" int wfx_stiffness_apply_part(wfx_stiffness* op, const void* x, const void* scale, void* y,
                                        int beta, int part, void* stream)
{
  WFX_API_BEGIN
  if (!op) fail("stiffness operator is NULL");
  if (part < -1 || part > 1) fail("part must be -1, 0 or 1");
  if (op->mode == WFX_STIFF_CELL_COLOUR && part >= 0) fail("stiffness: parts need the brick kernel");
  if (op->ncells == 0 && part == 1) return 0;
  apply_any(op, x, scale, y, beta, stream, part);
  WFX_API_END
}

extern "C" int wfx_stiffness_apply_scaled(wfx_stiffness* op, const void* x, const void* scale,
                                          void* y, void* stream)
{
  WFX_API_BEGIN
  if (!scale) fail("stiffness: scale vector is NULL");
  apply_any(op, x, scale, y, 0, stream);
  WFX_API_END
}

extern "C" int wfx_stiffness_apply_ensemble(wfx_stiffness* op, int nv, const void* x, const void* scale, void* y,
                                            int beta, void* stream)
{
  WFX_API_BEGIN
  if (!op) fail("stiffness operator is NULL");
  if (op->nshared > 0)
    fail("stiffness ensemble apply: the operator has %lld rank-shared dofs (ensembles are single-rank)",
         (long long)op->nshared);
  if (!op->ens) fail("stiffness ensemble apply: the operator was created without WFX_STIFF_ENSEMBLE");
  if (nv < 1 || nv > WFX_ENSEMBLE_MAX) fail("stiffness ensemble apply: nv = %d outside [1, %d]", nv, WFX_ENSEMBLE_MAX);
  if (scale && beta) fail("stiffness ensemble apply: a scale needs beta == 0");
  if (!x || !y) fail("stiffness: NULL vector");
  if (x == y) fail("stiffness: x and y must not alias");
  if (op->ncells == 0)
  {
    if (!beta)
      WFX_CUDA(cudaMemsetAsync(y, 0, (size_t)op->ndofs * nv * (op->dtype == WFX_F64 ? 8 : 4), (cudaStream_t)stream));
    return 0;
  }
  ScopedDevice sd(op->ctx->device);
  if (op->dtype == WFX_F64)
    dispatch_ens<double>(op, nv, (const double*)x, (const double*)scale, (double*)y, beta, (cudaStream_t)stream);
  else
    dispatch_ens<float>(op, nv, (const float*)x, (const float*)scale, (float*)y, beta, (cudaStream_t)stream);
  WFX_API_END
}

extern "C" int wfx_stiffness_apply_host(wfx_stiffness* op, const void* x_host, void* y_host, int beta)
{
  WFX_API_BEGIN
  if (!op) fail("stiffness operator is NULL");
  if (!x_host || !y_host) fail("stiffness: NULL vector");
  ScopedDevice sd(op->ctx->device);
  const size_t nb = (size_t)op->ndofs * (op->dtype == WFX_F64 ? 8 : 4);
  if (op->d_hx.n < nb) op->d_hx.alloc(nb);
  if (op->d_hy.n < nb) op->d_hy.alloc(nb);
  WFX_CUDA(cudaMemcpyAsync(op->d_hx.p, x_host, nb, cudaMemcpyHostToDevice, 0));
  if (beta) WFX_CUDA(cudaMemcpyAsync(op->d_hy.p, y_host, nb, cudaMemcpyHostToDevice, 0));
  apply_any(op, op->d_hx.p, nullptr, op->d_hy.p, beta, nullptr);
  WFX_CUDA(cudaMemcpyAsync(y_host, op->d_hy.p, nb, cudaMemcpyDeviceToHost, 0));
  WFX_CUDA(cudaStreamSynchronize(0));
  WFX_API_END
}

extern "C" int wfx_stiffness_mass_apply_host(wfx_stiffness* op, wfx_mass* mass, const void* x_host,
                                             void* y_host)
{
  WFX_API_BEGIN
  if (!op || !mass) fail("NULL operator");
  if (!x_host || !y_host) fail("stiffness: NULL vector");
  ScopedDevice sd(op->ctx->device);
  const void* minv = nullptr;
  if (wfx_mass_inverse_diagonal(mass, &minv)) fail("%s", wfx_last_error());
  const size_t nb = (size_t)op->ndofs * (op->dtype == WFX_F64 ? 8 : 4);
  if (op->d_hx.n < nb) op->d_hx.alloc(nb);
  if (op->d_hy.n < nb) op->d_hy.alloc(nb);
  WFX_CUDA(cudaMemcpyAsync(op->d_hx.p, x_host, nb, cudaMemcpyHostToDevice, 0));
  apply_any(op, op->d_hx.p, minv, op->d_hy.p, 0, nullptr);
  WFX_CUDA(cudaMemcpyAsync(y_host, op->d_hy.p, nb, cudaMemcpyDeviceToHost, 0));
  WFX_CUDA(cudaStreamSynchronize(0));
  WFX_API_END
}

extern "C" int wfx_stiffness_mass_apply_host_batch(wfx_stiffness* op, wfx_mass* mass, int nvec,
                                                   const void* const* x_hosts, void* const* y_hosts)
{
  WFX_API_BEGIN
  if (!op || !mass) fail("NULL operator");
  if (nvec < 0 || (nvec > 0 && (!x_hosts || !y_hosts))) fail("bad vector list");
  for (int i = 0; i < nvec; ++i)
    if (!x_hosts[i] || !y_hosts[i]) fail("stiffness: NULL vector %d", i);
  if (nvec == 0) return 0;
  ScopedDevice sd(op->ctx->device);
  const void* minv = nullptr;
  if (wfx_mass_inverse_diagonal(mass, &minv)) fail("%s", wfx_last_error());
  const size_t nb = (size_t)op->ndofs * (op->dtype == WFX_F64 ? 8 : 4);
  if (!op->bs_h2d)
  {
    WFX_CUDA(cudaStreamCreateWithFlags(&op->bs_h2d, cudaStreamNonBlocking));
    WFX_CUDA(cudaStreamCreateWithFlags(&op->bs_cmp, cudaStreamNonBlocking));
    WFX_CUDA(cudaStreamCreateWithFlags(&op->bs_d2h, cudaStreamNonBlocking));
    for (int q = 0; q < 2; ++q)
      for (cudaEvent_t* e : {&op->ev_x[q], &op->ev_y[q], &op->ev_fx[q], &op->ev_fy[q]})
        WFX_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  }
  for (int q = 0; q < 2; ++q)
  {
    if (op->d_bx[q].n < nb) op->d_bx[q].alloc(nb);
    if (op->d_by[q].n < nb) op->d_by[q].alloc(nb);
  }
  // vector i: H2D on one stream, the fused apply on a second, D2H on a third; buffer pair i % 2, so
  // the copy-in of vector i+1 and the copy-out of vector i-1 run under the apply of vector i (PCIe is
  // full duplex: the steady state costs max(H2D, D2H) per vector instead of their sum)
  for (int i = 0; i < nvec; ++i)
  {
    const int q = i & 1;
    if (i >= 2) WFX_CUDA(cudaStreamWaitEvent(op->bs_h2d, op->ev_fx[q], 0)); // apply i-2 has read d_bx[q]
    WFX_CUDA(cudaMemcpyAsync(op->d_bx[q].p, x_hosts[i], nb, cudaMemcpyHostToDevice, op->bs_h2d));
    WFX_CUDA(cudaEventRecord(op->ev_x[q], op->bs_h2d));
    WFX_CUDA(cudaStreamWaitEvent(op->bs_cmp, op->ev_x[q], 0));
    if (i >= 2) WFX_CUDA(cudaStreamWaitEvent(op->bs_cmp, op->ev_fy[q], 0)); // copy-out i-2 has read d_by[q]
    apply_any(op, op->d_bx[q].p, minv, op->d_by[q].p, 0, op->bs_cmp);
    WFX_CUDA(cudaEventRecord(op->ev_y[q], op->bs_cmp));
    WFX_CUDA(cudaEventRecord(op->ev_fx[q], op->bs_cmp));
    WFX_CUDA(cudaStreamWaitEvent(op->bs_d2h, op->ev_y[q], 0));
    WFX_CUDA(cudaMemcpyAsync(y_hosts[i], op->d_by[q].p, nb, cudaMemcpyDeviceToHost, op->bs_d2h));
    WFX_CUDA(cudaEventRecord(op->ev_fy[q], op->bs_d2h));
  }
  WFX_CUDA(cudaStreamSynchronize(op->bs_d2h));
  WFX_CUDA(cudaStreamSynchronize(op->bs_cmp));
  WFX_API_END
}

extern "C" int wfx_stiffness_info(wfx_stiffness* op, int64_t* num_cells, int* num_dofs_per_cell,
                                  int64_t* ndofs, double* flops, double* bytes, int* ncolours,
                                  int* nlaunches)
{
  WFX_API_BEGIN
  if (!op) fail("stiffness operator is NULL");
  const double n = op->N, s = op->dtype == WFX_F64 ? 8 : 4;
  if (num_cells) *num_cells = op->ncells;
  if (num_dofs_per_cell) *num_dofs_per_cell = op->nd;
  if (ndofs) *ndofs = op->ndofs;
  // sum-factorised count: 2 x 3 contractions of n MACs per point + symmetric 3x3 apply
  if (flops) *flops = (double)op->ncells * (12.0 * n * n * n * n + 18.0 * n * n * n);
  // algorithmic bytes (DESIGN.md): symmetric G + int32 dofmap per cell point; x, 1/m, y once
  // (affine fast path: 6 scalars per CELL and no per-point dofmap)
  if (bytes)
    *bytes = op->affine ? (double)op->ncells * 6 * s + (double)op->ndofs * 3 * s
                        : (double)op->ncells * op->nd * (6 * s + 4) + (double)op->ndofs * 3 * s;
  const int nc = (op->mode == WFX_STIFF_CELL_COLOUR || (op->cell2 && !op->cell2_brick)) ? op->cplan.ncolours : op->ncolours;
  if (ncolours) *ncolours = nc;
  if (nlaunches) *nlaunches = (op->persistent && op->mode != WFX_STIFF_CELL_COLOUR) ? 1 : nc;
  WFX_API_END
}

extern "C" int wfx_stiffness_kernel_info(wfx_stiffness* op, int* variant, int* affine, int* mixed,
                                         int* regular_batches, int* batches, int64_t* smem_bytes)
{
  WFX_API_BEGIN
  if (!op) fail("stiffness operator is NULL");
  if (variant) *variant = op->mode == WFX_STIFF_CELL_COLOUR ? -1 : (op->cell2 ? (op->cell2_brick ? 4 : 3) : op->variant);
  if (affine) *affine = op->affine ? 1 : 0;
  if (mixed) *mixed = op->mixed ? 1 : 0;
  if (regular_batches) *regular_batches = op->n_regular;
  if (batches) *batches = op->nbatches;
  if (smem_bytes) *smem_bytes = op->cell2 ? 0 : (int64_t)(op->variant ? op->smem_bytes_reg : op->smem_bytes);
  WFX_API_END
}

extern "C" int wfx_stiffness_destroy(wfx_stiffness* op)
{
  WFX_API_BEGIN
  if (op)
  {
    ScopedDevice sd(op->ctx->device);
    delete op;
  }
  WFX_API_END
}
