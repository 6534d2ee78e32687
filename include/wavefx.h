/*
 * wavefx.h -- C ABI of the B200-native waveFEniCS hot path (libwavefx.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++ or torch types.
 * Each entry point names the reference interface it replaces (paths relative to
 * the reference repository root).  The C++ functor wrappers with the reference's
 * own call shape live in wave-fenics_b200/hpp/wavefx.hpp; the Python ctypes
 * binding in wave-fenics_b200/capi.py.  INTEGRATION.md shows the binding a
 * maintainer of the reference would add.
 *
 * Conventions
 *  - every function returns 0 on success, non-zero on failure; the message is
 *    available from wfx_last_error() (thread-local).  The reference throws
 *    std::runtime_error (common/cuda/array.hpp:15-17,33-35); the C++ wrappers
 *    rethrow.
 *  - "_host" pointers are host memory, "_dev" pointers are device memory on the
 *    context's GPU.  Vectors have the DOLFINx la::Vector layout
 *    [owned | ghosts], block size 1, scalar type = the operator's dtype.
 *  - operators accumulate like the reference: y += A x  (common/operators.hpp:104,197)
 *    unless beta == 0 is passed, which computes y = A x without reading y.
 *  - `stream` is a cudaStream_t passed as void*; all _dev calls are asynchronous
 *    on it and never synchronise the device (the reference synchronises after
 *    every gather/scatter, common/cuda/scatter.cu:54,64).
 *  - there is no CPU fallback: without a usable GPU every device call fails.
 */
#ifndef WAVEFX_H
#define WAVEFX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WFX_VERSION 100

enum { WFX_F64 = 0, WFX_F32 = 1 };

/* stiffness kernel selection (wfx_stiffness_create flags) */
enum {
  WFX_STIFF_AUTO = 0,       /* brick-batched kernel when the plan supports it */
  WFX_STIFF_CELL_COLOUR = 1, /* simple per-cell kernel, coloured cells, global read-modify-write */
  WFX_STIFF_NO_SPLIT = 2,    /* (or-ed in) distributed meshes: do not schedule the interface batches as
                                a part of their own; the apply is then one pass and the ghost reduction
                                follows it (best when the reduction is cheap: NVLink peer memory) */
  WFX_STIFF_CELL_STREAM = 4, /* streamed-cell kernel: coloured cells, software-pipelined gather, FIRST / LAST
                                flags in the per-point dofmap (fused scaling, no memset); single-rank meshes.
                                WFX_STIFF_AUTO takes it by itself at the degrees where it measured faster */
  WFX_STIFF_ENSEMBLE = 8     /* (or-ed in) also build the ensemble path (wfx_stiffness_apply_ensemble); costs
                                at most one more per-point dofmap (4 B per cell point), no copy of G */
};

/* most fields of one ensemble */
#define WFX_ENSEMBLE_MAX 8

typedef struct wfx_ctx wfx_ctx;
typedef struct wfx_geom wfx_geom;
typedef struct wfx_stiffness wfx_stiffness;
typedef struct wfx_mass wfx_mass;
typedef struct wfx_boundary wfx_boundary;
typedef struct wfx_scatter_plan wfx_scatter_plan;
typedef struct wfx_comm wfx_comm;
typedef struct wfx_halo wfx_halo;
typedef struct wfx_wave wfx_wave;

const char* wfx_last_error(void);
int wfx_version(void);

/* ---- host-side tables: no GPU needed -------------------------------------- */

/* GLL points/weights on [0,1], n = P+1 per direction, ordering [0, 1, interior...]
 * = basix::quadrature::make_quadrature(gll, ...) as used at
 * common/precomputation.hpp:48-51, common/operators.hpp:16-19 (one direction). */
int wfx_gll(int P, double* pts, double* wts);

/* 1-D derivative matrix D[q*n+i] = l_i'(x_q), clamped like common/operators.hpp:26-29. */
int wfx_deriv_1d(int P, double* D);

/* tensor index -> DOLFINx local dof: compute_permutations (common/precompute.hpp:192-199),
 * = second member of tabulate_basis_and_permutation (common/operators.hpp:24). perm[(P+1)^3]. */
int wfx_compute_permutations(int P, int32_t* perm);

/* tabulate_basis_and_permutation (common/operators.hpp:13-32): table[4][nq][nd] (basis, d/dX0,
 * d/dX1, d/dX2 at the GLL points; dofs in DOLFINx order, points in the quadrature's tensor order,
 * entries clamped as at :26-29) and perm[nd].  Either output may be NULL.  The GPU operators never
 * form this dense table; it is exported for callers of the reference function. */
int wfx_tabulate_basis_and_permutation(int P, double* table, int32_t* perm);

/* reorder_dofmap (common/permute.hpp:10-28): out[c*nd+t] = in[c*nd+perm[t]]. */
int wfx_reorder_dofmap(int P, int64_t ncells, const int32_t* in_host, int32_t* out_host);

/* tabulate_1d (common/precompute.hpp:179-189): derivative-th derivative (0 or 1) of the
 * degree-P GLL Lagrange basis at the m=(q+2)/2 Gauss-Jacobi(0,0) points of degree q.
 * table[m][P+1]; returns m in *npoints (pass table = NULL to query). */
int wfx_tabulate_1d(int P, int q, int derivative, double* table, int* npoints);

/* ---- device context ------------------------------------------------------- */

/* replaces utils::set_device (common/cuda/utils.hpp:22-38): one context per GPU. */
int wfx_ctx_create(int device, wfx_ctx** ctx);
int wfx_ctx_destroy(wfx_ctx* ctx);
int wfx_ctx_sync(wfx_ctx* ctx);

/* raw device buffers: cuda::array<T> (common/cuda/array.hpp:8-51) as C calls */
int wfx_malloc(wfx_ctx* ctx, int64_t nbytes, void** ptr_dev);
int wfx_free(wfx_ctx* ctx, void* ptr_dev);
int wfx_memcpy_h2d(wfx_ctx* ctx, void* dst_dev, const void* src_host, int64_t nbytes);
int wfx_memcpy_d2h(wfx_ctx* ctx, void* dst_host, const void* src_dev, int64_t nbytes);

/* ---- geometry: precompute_geometric_data (common/precomputation.hpp:18-110) --
 * x_host [npts][3] (geometry.x()), xdofs_host [ncells][8] (geometry.dofmap(), P1 hex,
 * vertex v = ix + 2 iy + 4 iz).  Computes on the GPU, for every cell and GLL point,
 * detJ*w (with fabs, :95) and G = J^-1 (detJ w) J^-T clamped to -1/0/1 (:105-107),
 * in fp64, and keeps them on the device in the kernel's layout (symmetric 6-entry G)
 * in `dtype`. */
int wfx_geometry_create(wfx_ctx* ctx, int P, int dtype, int64_t ncells, int64_t npts,
                        const double* x_host, const int32_t* xdofs_host, wfx_geom** geom);
/* Copy back in the reference layout: G [ncells][nq][3][3], detJ [ncells][nq] (fp64;
 * either pointer may be NULL). */
int wfx_geometry_get(wfx_geom* geom, double* G_host, double* detJ_host);
/* n_affine: cells whose G is w_q times one constant matrix to rounding (parallelepipeds, detected from
 * the computed clamped G).  When every cell is affine the stiffness operator takes the structured
 * fast path: 6 scalars per CELL instead of 6 per point, the per-point array is never read. */
int wfx_geometry_info(wfx_geom* geom, int64_t* ncells, int64_t* n_affine);
/* Heterogeneous medium: multiplies the stored G of cell c by coeff_host[c] > 0, e.g.
 * (c0[c] / c0_ref)^2 so that a stiffness operator created with c0_ref applies -c0(x)^2 K with a
 * piecewise-constant speed of sound at no cost per apply.  The reference leaves this open
 * (`// TODO: Compute coefficients`, common/LinearGLL.hpp:170; `params` ignored at
 * common/operators.hpp:113-115).  The mass (detJ) is not touched.  Valid at any time before the applies
 * that should see it, on every kernel path: the private G copies stiffness operators made from this
 * geometry are scaled with it, and captured graphs keep their pointers.  Coefficients compose by
 * multiplication.  Synchronises the device; applies still in flight on other streams must have finished.
 * A refused coefficient (not positive, not finite) leaves G unchanged. */
int wfx_geometry_scale_cells(wfx_geom* geom, const double* coeff_host);
int wfx_geometry_destroy(wfx_geom* geom);

/* general-point building blocks of common/precompute.hpp (no fabs, no clamp, weights
 * applied by the caller), computed on the GPU, results returned to host arrays:
 *   compute_jacobian (:49-96)            J    [ncells][nq][3][3]
 *   compute_jacobian_determinant (:102)  detJ [ncells][nq]
 *   compute_jacobian_inverse (:122)      K    [ncells][nq][3][3]
 *   compute_geometrical_factor (:148)    G    [ncells][nq][3][3] = K K^T detJ w_q
 * points_host [nq][3]; weights_host [nq] (needed only when G_host != NULL);
 * any output pointer may be NULL. */
int wfx_compute_jacobian_data(wfx_ctx* ctx, int64_t ncells, int64_t npts, const double* x_host,
                              const int32_t* xdofs_host, int nq, const double* points_host,
                              const double* weights_host, double* J_host, double* detJ_host,
                              double* K_host, double* G_host);

/* ---- stiffness: StiffnessOperator (common/operators.hpp:136-201) -----------
 * dofmap_host: V->dofmap()->list().array(), [ncells][(P+1)^3] in DOLFINx local order
 * (the operator permutes to tensor order itself, like reorder_dofmap).  ndofs = number
 * of local vector entries (owned + ghosts).  c0: the reference hard-codes 1500
 * (operators.hpp:114) -- pass that for parity.  apply: y (+)= -c0^2 K x. */
int wfx_stiffness_create(wfx_ctx* ctx, wfx_geom* geom, int64_t ndofs, const int32_t* dofmap_host,
                         double c0, int flags, wfx_stiffness** op);
int wfx_stiffness_apply(wfx_stiffness* op, const void* x_dev, void* y_dev, int beta, void* stream);
/* Distributed meshes (one rank per GPU, GhostMode::none as demo/cpu_planar3d/main.cpp:42):
 * shared_dofs_host lists the local vector entries that also live on another rank (the union
 * of the halo's send and receive indices).  Cells touching them are scheduled first
 * (part 0, "interface"), the rest is part 1 ("interior"), so that the ghost reduction of
 * part 0's result can overlap part 1:  apply_part(.., 0) ; halo on another stream ;
 * apply_part(.., 1).  The fused scaling of wfx_stiffness_apply_scaled is then applied to
 * non-shared dofs only; shared dofs are scaled by wfx_halo_update_rev_fwd_scaled after
 * their sum is complete.  part = -1 runs both parts.  Part 1 continues the apply that the
 * preceding part-0 call on the same stream started: same x_dev / y_dev, x unchanged in between
 * (its first kernel may start while part 0 is still draining).  The operator keeps no per-apply
 * state: different streams may apply it concurrently (to different y). */
int wfx_stiffness_create_partitioned(wfx_ctx* ctx, wfx_geom* geom, int64_t ndofs,
                                     const int32_t* dofmap_host, double c0, int flags,
                                     int64_t nshared, const int32_t* shared_dofs_host,
                                     wfx_stiffness** op);
int wfx_stiffness_apply_part(wfx_stiffness* op, const void* x_dev, const void* scale_dev,
                             void* y_dev, int beta, int part, void* stream);
/* Fused operator+mass-inverse apply, the headline "stiffness + mass apply":
 *   y = scale .* (-c0^2 K x)   with scale_dev = 1/m (wfx_mass_inverse_diagonal).
 * Replaces stiff_op(u_n, b) followed by b/m (common/LinearGLL.hpp:173-191). */
int wfx_stiffness_apply_scaled(wfx_stiffness* op, const void* x_dev, const void* scale_dev,
                               void* y_dev, void* stream);
/* Ensemble apply: nv fields (1 <= nv <= WFX_ENSEMBLE_MAX) that share the mesh, the operator and c0, in
 * one pass over G and the dofmap.  Vectors are member-interleaved, [ndofs][nv]: entry (dof i, member m)
 * at i*nv + m -- the DOLFINx blocked la::Vector with block size bs = nv.  For every member m
 *   y[:,m] (+)= scale .* (-c0^2 K x[:,m])
 * scale_dev: [ndofs] (one value per dof for all members, e.g. 1/m) or NULL; a scale needs beta == 0 (as
 * wfx_stiffness_apply_scaled).  Needs an operator created with WFX_STIFF_ENSEMBLE and without rank-shared
 * dofs.  Deterministic: results repeat bit for bit, and a member's result does not depend on the others
 * or on its position in the ensemble. */
int wfx_stiffness_apply_ensemble(wfx_stiffness* op, int nv, const void* x_dev, const void* scale_dev,
                                 void* y_dev, int beta, void* stream);
/* Same call shape as the reference functor on host la::Vector arrays: copies x (and y
 * when beta != 0) to the GPU, applies, copies y back.  Synchronous. */
int wfx_stiffness_apply_host(wfx_stiffness* op, const void* x_host, void* y_host, int beta);
/* The headline path end to end with HOST buffers: y = M^-1 (-c0^2 K x), x and y host
 * arrays (pinned or pageable); H2D copy of x, fused apply, D2H copy of y.  Synchronous. */
int wfx_stiffness_mass_apply_host(wfx_stiffness* op, wfx_mass* mass, const void* x_host,
                                  void* y_host);
/* The same for nvec host vectors (several right-hand sides, or one vector per time step of a
 * host-driven loop): y_i = M^-1 (-c0^2 K x_i).  Copy-in, apply and copy-out of consecutive vectors are
 * pipelined on three streams with two device buffer pairs, so that in the steady state a vector costs
 * max(H2D, D2H) instead of H2D + apply + D2H.  Use pinned host memory, or the copies serialise.
 * Synchronous: returns when every y_i is complete. */
int wfx_stiffness_mass_apply_host_batch(wfx_stiffness* op, wfx_mass* mass, int nvec,
                                        const void* const* x_hosts, void* const* y_hosts);
/* num_cells / num_dofs / num_quads / flops as on the GPU operator classes
 * (common/cuda/mass.hpp:68-71); bytes = algorithmic bytes per apply (DESIGN.md). */
int wfx_stiffness_info(wfx_stiffness* op, int64_t* num_cells, int* num_dofs_per_cell,
                       int64_t* ndofs, double* flops, double* bytes, int* ncolours,
                       int* nlaunches);
/* Which kernel the plan selected: variant -1 simple per-cell kernel, 0 generic brick kernel (staged
 * local dofmap), 1 regular-brick kernel (arithmetic positions), 2 the same with the conflict-free P4
 * layout, 3 / 4 the streamed-cell kernel in colour / brick-plan order (no shared-memory dof arrays; the
 * other outputs then describe its plan); affine = 1: structured fast path (6 scalars of G per cell, the per-point array is never
 * read); mixed = 1: regular batches and irregular batches run their own kernel (two launches per
 * colour). */
int wfx_stiffness_kernel_info(wfx_stiffness* op, int* variant, int* affine, int* mixed,
                              int* regular_batches, int* batches, int64_t* smem_bytes);
/* Destroy an operator before the geometry it was created on (it removes its G copy from the geometry). */
int wfx_stiffness_destroy(wfx_stiffness* op);

/* ---- mass: MassOperatorCPU (common/operators.hpp:43-109) / SpectralMassOperator
 * (common/cuda/spectral_mass.hpp:23-99).  Collocated GLL => diagonal:
 *   y[i] (+)= (sum over cells c, points t with dof(c,perm[t]) == i of detJ[c,t]) * x[i]
 * The diagonal is reduced once at create time in the reference's cell order
 * (atomic-free segmented reduction). */
int wfx_mass_create(wfx_ctx* ctx, wfx_geom* geom, int64_t ndofs, const int32_t* dofmap_host,
                    wfx_mass** op);
int wfx_mass_apply(wfx_mass* op, const void* x_dev, void* y_dev, int beta, void* stream);
int wfx_mass_apply_host(wfx_mass* op, const void* x_host, void* y_host, int beta);
/* device pointers owned by the operator: m = M.1 (LinearGLL.hpp:102-110) and 1/m */
int wfx_mass_diagonal(wfx_mass* op, const void** m_dev);
int wfx_mass_inverse_diagonal(wfx_mass* op, const void** minv_dev);
/* y = x ./ m  (the b/m of common/LinearGLL.hpp:188-191 with the reciprocal precomputed);
 * x and y may alias. */
int wfx_mass_apply_inverse(wfx_mass* op, const void* x_dev, void* y_dev, void* stream);
/* Distributed meshes: sum the per-rank partial diagonals over the ranks sharing a dof
 * (m.scatter_rev(add), LinearGLL.hpp:110, followed by a forward update so that ghost copies
 * hold the assembled value too) and recompute 1/m.  Call once after wfx_mass_create. */
int wfx_mass_assemble(wfx_mass* op, wfx_halo* halo_f64);
int wfx_mass_destroy(wfx_mass* op);

/* ---- dofmap gather / scatter-add: gather<T>, scatter<T> (common/cuda/scatter.cu:47-65) */
/* out[i] = in[idx[i]], i < n */
int wfx_gather(wfx_ctx* ctx, int dtype, int64_t n, const int32_t* idx_dev, const void* in_dev,
               void* out_dev, void* stream);
/* atomic-free scatter-add plan for a fixed index array idx_host[n] into a vector of
 * length nout: out[j] (+)= sum_{i: idx[i]==j} in[i], contributions added in increasing i
 * (the order of the reference's serial loops), one thread per output entry. */
int wfx_scatter_plan_create(wfx_ctx* ctx, int64_t n, const int32_t* idx_host, int64_t nout,
                            wfx_scatter_plan** plan);
int wfx_scatter_add(wfx_scatter_plan* plan, int dtype, const void* in_dev, void* out_dev,
                    int beta, void* stream);
int wfx_scatter_plan_destroy(wfx_scatter_plan* plan);

/* ---- boundary linear form L (demo/cpu_planar3d/forms.ufl:21-24, assembled at
 * common/LinearGLL.hpp:175):  b += c0^2 g m1 - c0 m2 .* v_n  on facet dofs, with
 * m_tag the GLL-collocated facet mass of the facets carrying tag 1 / 2.
 * facets: (cell, local facet 0..5, tag) triplets -- the content of the MeshTags the
 * reference passes to create_form (LinearGLL.hpp:113-115). */
int wfx_boundary_create(wfx_ctx* ctx, int P, int dtype, int64_t nfacets,
                        const int32_t* facet_cell_host, const int32_t* facet_local_host,
                        const int32_t* facet_tag_host, int64_t npts, const double* x_host,
                        const int32_t* xdofs_host, int64_t ndofs, const int32_t* dofmap_host,
                        wfx_boundary** op);
int wfx_boundary_apply(wfx_boundary* op, double c0, double g, const void* vn_dev, void* b_dev,
                       void* stream);
/* dense copies of m1 / m2 (length ndofs, fp64) for checks */
int wfx_boundary_get(wfx_boundary* op, double* m1_host, double* m2_host);
/* Distributed meshes: sum the facet masses over the ranks sharing a boundary dof (fp64 halo), so
 * that every copy of the dof can add the complete boundary term after the ghost reduction. */
int wfx_boundary_assemble(wfx_boundary* op, wfx_halo* halo_f64);
int wfx_boundary_destroy(wfx_boundary* op);

/* ---- ghost-dof halo exchange: VectorUpdater (demo/gpu_scatter_mpi/VectorUpdater.hpp:21-230)
 * on NCCL instead of CUDA-aware MPI.  One process per GPU; the 128-byte id comes from
 * rank 0 (wfx_comm_unique_id) and is distributed by the caller (torch.distributed /
 * MPI_Bcast). */
int wfx_comm_unique_id(char id[128]);
int wfx_comm_create(wfx_ctx* ctx, const char id[128], int nranks, int rank, wfx_comm** comm);
int wfx_comm_destroy(wfx_comm* comm);
/* Index data as VectorUpdater reads it from the IndexMap (:31-59):
 *   fwd_send_*: per destination rank, the owned local indices whose values ghosts elsewhere
 *               mirror (scatter_fwd_indices + offsets);
 *   fwd_recv_*: per source rank, the local ghost positions (>= size_local) filled from it.
 * size_local / num_ghosts: the index map's sizes; offsets, ranks and every index are validated
 * against them on the host (send indices in [0, size_local), receive indices in the ghost part,
 * every ghost slot filled by one owner).  Collective over the communicator.
 * update_fwd: owner -> ghost copy (:132-143).  update_rev: ghost -> owner add (:189-199),
 * contributions added in neighbour order (atomic-free).  update_rev_fwd: the two fused,
 * one NCCL group each, leaving every copy of a shared dof bitwise identical. */
int wfx_halo_create(wfx_ctx* ctx, wfx_comm* comm, int dtype, int64_t size_local, int64_t num_ghosts,
                    int n_send_nbr, const int32_t* send_ranks, const int32_t* send_offsets,
                    const int32_t* send_indices, int n_recv_nbr, const int32_t* recv_ranks,
                    const int32_t* recv_offsets, const int32_t* recv_indices, wfx_halo** halo);
/* 1: the fused ghost reduction runs over NVLink peer memory (one kernel that writes the neighbours'
 * receive buffers directly), 0: over NCCL send/recv groups.  Peer memory is chosen when every rank
 * of the communicator is a process on this host with a peer-accessible GPU; the environment
 * variable WFX_HALO_TRANSPORT = auto | nccl | p2p overrides (p2p: fail instead of falling back). */
int wfx_halo_transport(wfx_halo* halo, int* transport);
int wfx_halo_update_fwd(wfx_halo* halo, void* x_dev, void* stream);
int wfx_halo_update_rev(wfx_halo* halo, void* x_dev, void* stream);
int wfx_halo_update_rev_fwd(wfx_halo* halo, void* x_dev, void* stream);
/* as update_rev_fwd, the owner multiplying the completed sum by scale_dev[i] before it is sent
 * back to the ghosts (the b/m of common/LinearGLL.hpp:188-191 for shared dofs) */
int wfx_halo_update_rev_fwd_scaled(wfx_halo* halo, void* x_dev, const void* scale_dev, void* stream);
int wfx_halo_destroy(wfx_halo* halo);

/* ---- wave model + RK4: LinearGLLOpt (common/LinearGLL.hpp:37-287) ----------
 * Borrows the operators (they must outlive the model).  halo may be NULL (one rank).
 * size_local: number of owned dofs (axpy touches owned entries only, :30).
 * State vectors u_n, v_n live on the device in the operators' dtype.
 * Distributed meshes: halo must have the model's dtype.  The lumped mass and the facet masses are
 * summed over the ranks here when the model is fp64; an fp32 model must have them assembled
 * beforehand (wfx_mass_assemble / wfx_boundary_assemble with a separate fp64 halo) or create fails. */
int wfx_wave_create(wfx_ctx* ctx, wfx_stiffness* stiff, wfx_mass* mass, wfx_boundary* bnd,
                    wfx_halo* halo, int64_t size_local, double c0, double f0, double p0,
                    wfx_wave** wave);
/* Ensemble model: nv members (1 <= nv <= WFX_ENSEMBLE_MAX) on one rank that share the mesh, the operators
 * and c0; member m is the model LinearGLLOpt(..., c0, f0_host[m], p0_host[m]) with its own source
 * g_m(t) = window_m(t) p0_m w_m / c0 cos(w_m t), w_m = 2 pi f0_m, and its own four-period Hann ramp.
 * stiff must have been created with WFX_STIFF_ENSEMBLE.  init, set_state, get_state, state_ptrs, f0, f1,
 * rk4, set_probes, get_probe_series, set_field_stats, get_field_stats and destroy accept the model; their vectors are then
 * member-interleaved [ndofs][nv] (see wfx_stiffness_apply_ensemble), probe values [nrecords][nprobes][nv].
 * set_snapshot refuses an ensemble model. */
int wfx_wave_create_ensemble(wfx_ctx* ctx, wfx_stiffness* stiff, wfx_mass* mass, wfx_boundary* bnd, int nv,
                             int64_t size_local, double c0, const double* f0_host, const double* p0_host,
                             wfx_wave** wave);
/* Lossy (beta == 0) and Westervelt (beta > 0) models on one rank (DESIGN.md section 4.5a).  Pressure p:
 *   (1 - kappa p) p_tt - c0^2 lap p - delta lap p_t = kappa p_t^2,   kappa = 2 beta / (rho0 c0^2)
 *   dp/dn = g(t) on tag 1 (g as in wfx_wave_create), dp/dn = -p_t / c0 on tag 2.
 * Lumped GLL system per dof i, with s = delta / c0^2 and q = (delta / c0) m2:
 *   (m_i (1 - kappa p_i) + q_i) p_tt,i = [-c0^2 K (p + s p_t)]_i + kappa m_i p_t,i^2
 *                                        + (c0^2 g + delta g') m1_i - c0 m2_i p_t,i
 * (the stiffness term uses the operator's own c0: -delta K p_t exactly).  delta = beta = 0 is
 * wfx_wave_create's model, bit for bit.  With wfx_geometry_scale_cells the per-cell coefficient multiplies
 * the delta term too: delta_eff(x) = delta coeff(x).
 * delta >= 0 [m^2/s], beta >= 0, rho0 > 0 [kg/m^3] when beta > 0, f0 > 0, all finite; the stiffness operator
 * must have no rank-shared dofs.  init / set_state / get_state / state_ptrs / f0 / f1 / rk4 / probes /
 * snapshots / destroy accept the model (single-field vectors). */
int wfx_wave_create_westervelt(wfx_ctx* ctx, wfx_stiffness* stiff, wfx_mass* mass, wfx_boundary* bnd,
                               int64_t size_local, double c0, double f0, double p0, double delta, double beta,
                               double rho0, wfx_wave** wave);
int wfx_wave_init(wfx_wave* wave);                                   /* :131-134 */
/* Copies the state to the device; on a distributed mesh the ghost entries are then overwritten by
 * their owners' values (u->scatter_fwd(), v->scatter_fwd(), :164,167). */
int wfx_wave_set_state(wfx_wave* wave, const void* u_host, const void* v_host);
int wfx_wave_get_state(wfx_wave* wave, void* u_host, void* v_host);
int wfx_wave_state_ptrs(wfx_wave* wave, void** u_dev, void** v_dev);
/* The right-hand sides on their own, device vectors of ndofs entries (dtype of the model):
 *   f0(t, u, v, result): result = v                                  (:141-144)
 *   f1(t, u, v, result): result = M^-1 (-c0^2 K u + boundary(g(t), v)) (:151-192), including the
 *   ghost reduction on a distributed mesh.  result must not alias u or v.
 *   Precondition on a distributed mesh: the ghost entries of u and v equal their owners' values
 *   (the reference calls scatter_fwd on its own u, v first, :164,167; here u and v are the caller's
 *   const vectors -- wfx_halo_update_fwd them if in doubt). */
int wfx_wave_f0(wfx_wave* wave, double t, const void* u_dev, const void* v_dev, void* result_dev,
                void* stream);
int wfx_wave_f1(wfx_wave* wave, double t, const void* u_dev, const void* v_dev, void* result_dev,
                void* stream);
/* rk4(startTime, finalTime, timeStep) (:198-287).  max_steps <= 0: run to tf.
 * Returns steps taken and the final time. */
int wfx_wave_rk4(wfx_wave* wave, double t0, double tf, double dt, int64_t max_steps,
                 int64_t* steps, double* t_end, void* stream);
/* ---- solution output (the reference has none: it prints the solve time only,
 * demo/cpu_planar3d/main.cpp:87-93) ------------------------------------------------------------
 * Probes: after every completed time step the values u[dofs] are appended to a series kept on the
 * device (at most max_records steps; later steps are not recorded).  get_probe_series copies the
 * recorded times (the t reached after each step) and values [nrecords][nprobes] (model dtype) to the
 * host; either pointer may be NULL.  init / set_state start a new series. */
int wfx_wave_set_probes(wfx_wave* wave, int64_t nprobes, const int32_t* dofs_host, int64_t max_records);
int wfx_wave_get_probe_series(wfx_wave* wave, int64_t* nrecords, double* t_host, void* values_host);
/* Field statistics (DESIGN.md section 4.5b): maps of the pressure u over the steady-state part of a run,
 * accumulated on the device.  After every completed time step whose reached time t_n satisfies
 * t_n >= t_start - dt_step / 2 (dt_step: the size of that step), every local entry i (owned and ghost;
 * every member of an ensemble) is sampled:
 *   pmax[i] = max_n u_i(t_n), pmin[i] = min_n u_i(t_n)   (model dtype, NaN propagates)
 *   harm_h[i] = (2 / N) sum_n u_i(t_n) exp(-i h w t_n),   h = 1..nharm, w = 2 pi f0 (member m: f0_host[m]),
 * accumulated in fp64 for both model dtypes, N the number of sampled steps.  With whole periods in the window
 * and whole steps per period, Re(harm_h e^{i h w t}) is the h-th Fourier component of the sampled signal.
 * init, set_state and set_field_stats reset the accumulators; a run split across several rk4 calls keeps
 * accumulating.  Probes and snapshots are independent of them.
 * enable = 0 switches off and frees the accumulators.  Otherwise allocates/resets them:
 * pmax/pmin in the model dtype, H complex fp64 accumulators, all [ndofs] or [ndofs][nv].
 * nharm in [0, WFX_HARMONICS_MAX], t_start finite. */
#define WFX_HARMONICS_MAX 8
int wfx_wave_set_field_stats(wfx_wave* wave, int enable, double t_start, int nharm);
/* Synchronises like wfx_wave_get_probe_series.  nsamples = N, t_first/t_last = first and last sampled time;
 * pmax_host/pmin_host in the model dtype (member-interleaved for ensembles); harm_host complex128
 * [nharm][ndofs*nv] as (re, im) pairs, already scaled by 2/N.  Any output pointer may be NULL.
 * N = 0: pmax = -inf, pmin = +inf, harmonics 0 (t_first = t_last = 0).  Refused when the statistics are off. */
int wfx_wave_get_field_stats(wfx_wave* wave, int64_t* nsamples, double* t_first, double* t_last,
                             void* pmax_host, void* pmin_host, double* harm_host);
/* The statistics' current settings: enabled (0 / 1), t_start and nharm (0 when off), e.g. to size the buffers of
 * wfx_wave_get_field_stats.  Any output pointer may be NULL. */
int wfx_wave_field_stats_info(wfx_wave* wave, int* enabled, double* t_start, int* nharm);
/* Source profile (DESIGN.md section 4.5c): phased-array sources on the tag-1 facets.  With a profile, the
 * boundary term of every model uses per-entry delayed sources in place of g(t):
 *   g_i(t) = a_i g(t - tau_i),   g(s) = g'(s) = 0 for s < 0,
 * g the model's source including its four-period ramp (lossy / Westervelt models: a_i (g + (delta / c0^2) g')
 * (t - tau_i); ensemble member m: its own f0 / p0).  The sources are evaluated on the device in fp64 at every
 * stage time, for both model dtypes.  amp_host and delay_host hold the model's local entries in the state
 * layout (ndofs, or ndofs * nv member-interleaved for an ensemble); entries off tag 1 are ignored.  Either may be
 * NULL (a = 1, tau = 0 respectively); both NULL clears the profile and restores the unprofiled path.
 * The profile is model configuration: it survives init, set_state and snapshot restarts, and may be changed
 * between rk4 calls.  Refused: a NULL model, a model without a boundary operator, a distributed model, a
 * non-finite amplitude or delay, a negative delay. */
int wfx_wave_set_source_profile(wfx_wave* wave, const double* amp_host, const double* delay_host);
/* Snapshots / checkpoints: every `every` completed steps (counted since init / set_state) u and v are
 * copied device -> device on the stepping stream and device -> pinned host on a separate copy stream
 * while the time stepping continues; `fn` then receives host pointers valid for the duration of the
 * call (step number, time reached, u, v in the model dtype, ndofs entries each).  It runs on the
 * thread that called wfx_wave_rk4, at the next snapshot or before rk4 returns.  A checkpoint is a
 * snapshot fed back through wfx_wave_set_state.  every = 0 or fn = NULL switches snapshots off. */
typedef void (*wfx_snapshot_fn)(void* user, int64_t step, double t, const void* u_host, const void* v_host);
int wfx_wave_set_snapshot(wfx_wave* wave, int64_t every, wfx_snapshot_fn fn, void* user);
int wfx_wave_destroy(wfx_wave* wave);

/* ---- thermal model: Pennes bioheat equation + RK4 with a CEM43 thermal dose (DESIGN.md section 4.5d) ------
 * State: the temperature rise theta = T - T_art over the arterial temperature, in the operators' dtype.
 *   rhoC theta_t = div(k grad theta) - wbCb theta + s Q            in the domain
 *   -k d theta / dn = h_j (theta - (T_ext_j - T_art))              on the tag-j facets, j = 1, 2
 * all other faces insulated.  Lumped GLL system per dof i (m: lumped mass, m1 / m2: the facet masses of bnd):
 *   theta_i' = scale_i [-cK^2 K theta]_i - r_i theta_i + f_i,   scale_i = (k / cK^2) / (rhoC_i m_i)
 *   r_i = (wbCb_i m_i + h1 m1_i + h2 m2_i) / (rhoC_i m_i)
 *   f_i = (h1 m1_i (T_ext1 - T_art) + h2 m2_i (T_ext2 - T_art) + s Q_i m_i) / (rhoC_i m_i)
 * with cK the stiffness operator's c0, so that the diffusion term is one fused wfx_stiffness_apply_scaled.  A
 * per-cell conductivity k_c is the operator's geometry scaled by wfx_geometry_scale_cells(k_c / k) before the
 * stiffness operator is created.  The model borrows the operators (they must outlive it) and may share them with
 * a wave model whose geometry is unscaled.  One rank only.
 * k [W/(m K)] > 0; rhoc_host [ndofs] [J/(m^3 K)] > 0; perf_host [ndofs] (wbCb [W/(m^3 K)]) >= 0 or NULL (0);
 * h_host[2] [W/(m^2 K)] >= 0 or NULL (insulated); T_ext_host[2] or NULL (T_art); h != 0 needs bnd.  All finite.
 * Per-cell rhoC and wbCb enter as mass-weighted averages sum_c coeff_c (detJ w)_{c,i} / m_i (INTEGRATION.md).
 * The heat source Q starts at 0 and the heat scale s at 1.
 *
 * Dose: after every completed step of size dt_n, with T_i = T_art + theta_i at its end,
 *   CEM43_i += (dt_n / 60) R^(43 - T_i),  R = 0.5 for T_i >= 43, else 0.25   (fp64; t in s, CEM43 in min)
 *   theta_max_i = max(theta_max_i, theta_i)                                  (model dtype, NaN propagates)
 * init and set_state reset both (CEM43 = 0, theta_max = -inf) and the step count; a run split over several rk4
 * calls keeps accumulating. */
typedef struct wfx_thermal wfx_thermal;
int wfx_thermal_create(wfx_ctx* ctx, wfx_stiffness* stiff, wfx_mass* mass, wfx_boundary* bnd, double k,
                       const double* rhoc_host, const double* perf_host, double T_art, const double* h_host,
                       const double* T_ext_host, wfx_thermal** th);
int wfx_thermal_init(wfx_thermal* th); /* theta = 0 */
int wfx_thermal_set_state(wfx_thermal* th, const void* theta_host);
int wfx_thermal_get_state(wfx_thermal* th, void* theta_host);
int wfx_thermal_state_ptr(wfx_thermal* th, void** theta_dev);
/* Q [W/m^3] per dof, fp64; NULL: Q = 0.  Non-finite values are refused. */
int wfx_thermal_set_heat_source(wfx_thermal* th, const double* q_host);
/* Q from the harmonic maps of a wave model's field statistics (wfx_wave_set_field_stats), on the device:
 *   Q_i = sum_{h=1..H} alpha_i(h f0_m) |p_h,i|^2 / (rho0 c0),   alpha_i(f) = alpha0_i (f / 1 MHz)^y  [Np/m]
 * with p_h = (2 / N) times the accumulated sums (as wfx_wave_get_field_stats scales them), member m's amplitudes
 * and source frequency f0_m (m = 0 for a single-field model).  alpha0_host [ndofs] or NULL (alpha0 everywhere).
 * Refused: statistics off, N = 0 or H = 0, member out of range, a wave on another context or with another ndofs,
 * alpha0 < 0, rho0 <= 0, c0 <= 0 or non-finite parameters. */
int wfx_thermal_heat_from_wave(wfx_thermal* th, wfx_wave* wave, int member, double alpha0,
                               const double* alpha0_host, double y, double rho0, double c0);
int wfx_thermal_get_heat_source(wfx_thermal* th, double* q_host);
/* s >= 0, finite: duty cycles; heating then cooling is two rk4 calls with s = 1 and s = 0 */
int wfx_thermal_set_heat_scale(wfx_thermal* th, double s);
/* out = theta' at theta (device vectors of ndofs entries, model dtype); out must not alias theta */
int wfx_thermal_rhs(wfx_thermal* th, const void* theta_dev, void* out_dev, void* stream);
/* classical RK4 from t0 to tf (loop of wfx_wave_rk4: while t < tf, dt = min(dt, tf - t)); max_steps <= 0: run
 * to tf.  Graph replay on one rank as wfx_wave_rk4 (WFX_WAVE_GRAPH=0 switches it off). */
int wfx_thermal_rk4(wfx_thermal* th, double t0, double tf, double dt, int64_t max_steps, int64_t* steps,
                    double* t_end, void* stream);
/* steps since init / set_state; cem43_host [ndofs] fp64, theta_max_host [ndofs] model dtype; any may be NULL */
int wfx_thermal_get_dose(wfx_thermal* th, int64_t* nsteps, double* cem43_host, void* theta_max_host);
/* Power iteration (iters >= 1 applications, deterministic) for the largest eigenvalue lambda of theta -> -theta'
 * without its source (self-adjoint in the rhoC m inner product), estimated by the Rayleigh quotient, and
 * dt_max = 2.785293563405282 / lambda, the RK4 stability limit on the negative real axis.  The estimate
 * approaches lambda from below, so dt_max is an upper bound's estimate: step with a safety factor (e.g. 0.8). */
int wfx_thermal_stable_dt(wfx_thermal* th, int iters, double* lambda, double* dt_max);
int wfx_thermal_destroy(wfx_thermal* th);

#ifdef __cplusplus
}
#endif
#endif /* WAVEFX_H */
