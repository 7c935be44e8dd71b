/* pmgx.h -- C ABI of the B200-native p-multigrid hot path (drop-in boundary).
 *
 * Every entry point replaces one piece of the reference's header-only C++
 * operator API (Wells-Group/pmg-dolfinx, paths relative to the reference root);
 * the reference interface each one stands in for is cited next to it.  The C++
 * shim include/pmgx/dolfinx_acc_compat.hpp re-creates the reference's class
 * names and method signatures on top of these functions.
 *
 * Conventions
 *   - every function returns 0 on success, a PMGX_ERR_* code otherwise;
 *     pmgx_last_error_string() describes the last failure of the calling thread;
 *   - pointer arguments are DEVICE pointers unless the name ends in _h (host);
 *   - vectors follow the reference layout: owned entries [0, n_owned) first,
 *     ghosts after (src/vector.hpp:86,213-225); all scalars are FP64, indices
 *     int32, BC markers int8;
 *   - caller arrays handed to *_create are borrowed for the handle's lifetime
 *     unless stated otherwise; *_destroy frees everything the handle owns;
 *   - all device work is enqueued on the context's compute stream and is
 *     asynchronous w.r.t. the host unless a host scalar is returned;
 *   - there is NO CPU fallback: every compute entry point fails with
 *     PMGX_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef PMGX_H
#define PMGX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMGX_OK 0
#define PMGX_ERR_ARG 1
#define PMGX_ERR_CUDA 2
#define PMGX_ERR_NCCL 3
#define PMGX_ERR_NUMERIC 4
#define PMGX_ERR_UNSUPPORTED 5

#define PMGX_MAX_DEGREE 8
#define PMGX_NCCL_ID_BYTES 128

typedef struct pmgx_ctx pmgx_ctx;
typedef struct pmgx_halo pmgx_halo;
typedef struct pmgx_operator pmgx_operator;
typedef struct pmgx_cheb pmgx_cheb;
typedef struct pmgx_cg pmgx_cg;
typedef struct pmgx_interp pmgx_interp;
typedef struct pmgx_coarse pmgx_coarse;
typedef struct pmgx_vcycle pmgx_vcycle;
typedef struct pmgx_boxmesh pmgx_boxmesh;
typedef struct pmgx_ghostmesh pmgx_ghostmesh;
typedef struct pmgx_amg_hier pmgx_amg_hier;

/* ------------------------------------------------------------------ misc -- */
const char* pmgx_last_error_string(void);
int pmgx_version(void);

/* 1-D GLL tables the reference takes from Basix (src/laplacian.hpp:299-317,
 * src/precompute.hpp:255-271, src/interpolate.hpp:118).  Host, no GPU needed.
 *   points_h[n], weights_h[n] on [0,1]; dphi_h[n*n] row = quadrature point;
 *   interp_h[(pf+1)*(pc+1)] = l^c_ic(x^f_if). n = degree+1. Any pointer may be NULL. */
int pmgx_gll_tables(int degree, double* points_h, double* weights_h, double* dphi_h);
int pmgx_gll_interp_1d(int degree_coarse, int degree_fine, double* interp_h);

/* Eigenvalues of a symmetric tridiagonal matrix, QL with implicit shifts
 * (replaces tqli, src/cg.hpp:15-84).  d_h[n] in/out, e_h[n] in (destroyed). */
int pmgx_tqli(double* d_h, double* e_h, int n);

/* --------------------------------------------------------------- context -- */
/* One context per GPU / rank (replaces "one MPI rank per GPU",
 * examples/pmg/select_gpu.sh + MPI_COMM_WORLD).  nccl_id_h: PMGX_NCCL_ID_BYTES
 * from pmgx_nccl_unique_id() on rank 0 and broadcast by the launcher (torchrun /
 * torch.distributed, threads, ...); NULL iff nranks == 1. */
int pmgx_nccl_unique_id(void* id_h);
int pmgx_ctx_create(int device, int rank, int nranks, const void* nccl_id_h, pmgx_ctx** out);
int pmgx_ctx_destroy(pmgx_ctx* ctx);
int pmgx_ctx_sync(pmgx_ctx* ctx);                 /* device_synchronize, src/util.hpp:51-58 */
void* pmgx_ctx_stream(pmgx_ctx* ctx);             /* cudaStream_t of the compute stream */
int pmgx_ctx_rank(pmgx_ctx* ctx);
int pmgx_ctx_nranks(pmgx_ctx* ctx);
/* number of kernels launched by this library on ctx since creation (bench "gpu_launches") */
long long pmgx_ctx_launch_count(pmgx_ctx* ctx);
/* Per-kernel timing of the matrix-free apply kernel (bench roofline): while on, every launch of
 * the apply kernel is bracketed by CUDA events on the compute stream; _read synchronises and
 * returns the summed device time and the launch count for one degree, then clears them. */
/* 1 when the NVLink peer-memory path is active (nranks > 1, all ranks on one node, CUDA IPC
 * available, PMGX_P2P != 0): halo values and all-reduce operands are stored straight into the
 * peers' memory by the library's own kernels; 0: grouped ncclSend/ncclRecv + ncclAllReduce. */
int pmgx_ctx_uses_p2p(pmgx_ctx* ctx);
int pmgx_ctx_profile(pmgx_ctx* ctx, int on);
int pmgx_ctx_profile_read(pmgx_ctx* ctx, int degree, double* ms_total_h, long long* launches_h);

/* ------------------------------------------------------------------ halo -- */
/* Owner->ghost forward scatter plan (replaces dolfinx::common::Scatterer held by
 * acc::Vector, src/vector.hpp:83-95).  send_idx_h: owned local indices grouped by
 * destination rank (Scatterer::local_indices); recv_idx_h: ghost slot (0-based in
 * the ghost block) of each received value grouped by source rank
 * (Scatterer::remote_indices).  The index arrays are copied.  With nranks > 1 this call is
 * COLLECTIVE (like constructing a Scatterer on an MPI communicator): every rank must create its
 * halos in the same order, because the ranks exchange the IPC handles of their receive buffers. */
int pmgx_halo_create(pmgx_ctx* ctx, int n_owned, int n_ghost,
                     int n_send_nbr, const int* send_ranks_h, const int* send_offsets_h,
                     const int32_t* send_idx_h,
                     int n_recv_nbr, const int* recv_ranks_h, const int* recv_offsets_h,
                     const int32_t* recv_idx_h, pmgx_halo** out);
int pmgx_halo_destroy(pmgx_halo* h);
int pmgx_halo_uses_p2p(pmgx_halo* h);
/* Vector::scatter_fwd_begin / scatter_fwd_end (src/vector.hpp:186-238) on the comm stream:
 * peer-memory path: ONE kernel packs and stores into the neighbours' receive buffers over NVLink
 * and releases an epoch flag, a one-CTA kernel waits for the neighbours' flags, then unpack;
 * NCCL path: pack kernel + grouped ncclSend/ncclRecv + unpack.  The compute stream only waits
 * in _end. */
int pmgx_halo_fwd_begin(pmgx_halo* h, double* x);
int pmgx_halo_fwd_end(pmgx_halo* h, double* x);
/* Vector::scatter_rev (src/vector.hpp:249-294): ghost -> owner accumulate. */
int pmgx_halo_rev(pmgx_halo* h, double* x);
/* stand-alone gather/scatter kernels: pack / unpack / unpack_add, src/vector.hpp:24-55 */
int pmgx_pack(pmgx_ctx* ctx, int n, const int32_t* idx, const double* in, double* out);
int pmgx_unpack(pmgx_ctx* ctx, int n, const int32_t* idx, const double* in, double* out);
int pmgx_unpack_add(pmgx_ctx* ctx, int n, const int32_t* idx, const double* in, double* out);

/* ---------------------------------------------------------- vector kernels -- */
/* Free functions of dolfinx::acc (src/vector.hpp:333-454) on raw device arrays. */
int pmgx_vec_set(pmgx_ctx* ctx, double* x, long long n, double v);                 /* Vector::set :109 */
int pmgx_vec_copy(pmgx_ctx* ctx, double* a, const double* b, long long n);         /* copy :423 */
int pmgx_vec_axpy(pmgx_ctx* ctx, double* r, double alpha, const double* x,
                  const double* y, long long n);                                   /* axpy :397 r=alpha*x+y */
int pmgx_vec_scale(pmgx_ctx* ctx, double* r, double alpha, long long n);           /* scale :412 */
int pmgx_vec_pointwise_mult(pmgx_ctx* ctx, double* w, const double* x,
                            const double* y, long long n);                         /* pointwise_mult :437 */
int pmgx_vec_mask_bc(pmgx_ctx* ctx, double* b, const int8_t* bc, long long n);     /* b*=(1-bc) pmg.hpp:100-103 */
/* inner_product / squared_norm / norm (src/vector.hpp:333-390): local reduction over the
 * n owned entries + all-reduce over ranks; result returned on the host (blocking). */
int pmgx_vec_dot(pmgx_ctx* ctx, const double* a, const double* b, long long n, double* result_h);
int pmgx_vec_norm(pmgx_ctx* ctx, const double* a, long long n, int linf, double* result_h);

/* -------------------------------------------------- matrix-free Laplacian -- */
#define PMGX_LAP_DEFAULT 0
#define PMGX_LAP_LITERAL_DETJ 1   /* reproduce detJ of src/laplacian.hpp:97 verbatim (quirk Q17) */
#define PMGX_LAP_NO_DIAG 2        /* skip the matrix-free diagonal at create */
#define PMGX_LAP_STREAM_G 4       /* always stream the per-quadrature-point G (the reference's data flow,
                                     src/laplacian.hpp:221-227); default: when every cell of the operator is
                                     affine the apply uses one geometry 6-vector per cell, G(q) = w_q Gc */
#define PMGX_LAP_RECOMPUTE_G 8    /* keep no geometry: no per-quadrature-point G and no per-cell Gc.  Every apply,
                                     CSR assembly and get_G computes G from the borrowed xgeom / geom_dofmap (the
                                     reference's batch_size > 0 mode, src/laplacian.hpp:383-396), so vertices moved
                                     in place take effect at the next apply; the diagonal is still computed once at
                                     create.  No affinity test runs (is_affine() is 0); PMGX_LAP_STREAM_G has no
                                     effect with it; PMGX_LAP_LITERAL_DETJ and PMGX_LAP_NO_DIAG apply as usual. */
#define PMGX_LAP_GEOM_Q2 16       /* second-order (27-node, triquadratic) geometry: geom_dofmap[n_cells][27] and xgeom
                                     holds the geometry node coordinates.  Node k = 9a + 3b + c, a, b, c in {0, 1, 2}
                                     at reference coordinates {0, 1/2, 1} along (x, y, z): the lexicographic
                                     extension of the trilinear order 4a + 2b + c, with the 8 corners at k = 0, 2,
                                     6, 8, 18, 20, 24, 26.  G and det J are formed at the GLL points from the
                                     quadratic map.  A cell is affine when all 27 nodes sit at v000 + (a/2) e1 +
                                     (b/2) e2 + (c/2) e3 (tolerance 1e-13 of the longest edge); a mesh of such cells
                                     runs the same affine kernel as its 8-node form, any other mesh the streamed-G
                                     kernel.  PMGX_LAP_LITERAL_DETJ, PMGX_LAP_NO_DIAG and PMGX_LAP_STREAM_G keep their
                                     meaning; with PMGX_LAP_RECOMPUTE_G create fails with PMGX_ERR_UNSUPPORTED (the
                                     recompute apply kernels form trilinear Jacobians only). */

/* MatFreeLaplacian ctor (src/laplacian.hpp:289-349).  dofmap[n_cells][(P+1)^3],
 * xgeom[n_points][3], geom_dofmap[n_cells][8] (tensor-product vertex order; [n_cells][27] with
 * PMGX_LAP_GEOM_Q2),
 * kappa[n_cells] (read on every apply, like cell_constants :230), lcells_h/bcells_h:
 * host lists (src/mesh.hpp:105-143), bc_marker[n_owned+n_ghost].  The 1-D GLL table,
 * the trilinear geometry table and the weights (dphi_geometry / G_weights arguments of
 * the reference) are generated internally.  dofmap and bc_marker are snapshotted into
 * an internal BC-encoded copy in launch order; G is owned (reference :512). halo may be
 * NULL (single rank). */
int pmgx_laplacian_create(pmgx_ctx* ctx, int degree, int n_cells, const int32_t* dofmap,
                          const double* xgeom, int n_points, const int32_t* geom_dofmap,
                          const double* kappa, const int32_t* lcells_h, int n_lcells,
                          const int32_t* bcells_h, int n_bcells, const int8_t* bc_marker,
                          int n_owned, int n_ghost, pmgx_halo* halo, int flags,
                          pmgx_operator** out);
/* Geometry factors in the reference layout G[n_list][nq][6] (src/laplacian.hpp:99-111), list
 * order = lcells then bcells (:329-336); for parity tests against geometry_computation. */
int pmgx_laplacian_get_G(pmgx_operator* op, double* G_out);
/* 1 when the operator runs the affine-geometry kernel (all cells affine, no PMGX_LAP_STREAM_G) */
int pmgx_laplacian_is_affine(pmgx_operator* op);
/* name and template arguments of the apply kernel this operator launches (for bench / profiles) */
int pmgx_laplacian_kernel_name(pmgx_operator* op, char* name_h, int cap);
/* bytes of device memory the operator owns: launch-order permutation, encoded dofmap, G, Gc and the
 * inverse diagonal (for sizing problems, and to compare PMGX_LAP_RECOMPUTE_G against the default) */
int pmgx_laplacian_device_bytes(pmgx_operator* op, long long* bytes_h);

/* ------------------------------------------------------------- CSR operator -- */
/* MatrixOperator (src/csr.hpp:57-131): row_ptr[n_rows+1], off_diag_offset[n_rows] (first
 * ghost-column entry of each row), cols, values -- HOST arrays, copied.  Columns >= n_owned
 * address ghosts.  diag^-1 is extracted like src/csr.hpp:101-112. */
int pmgx_csr_create(pmgx_ctx* ctx, int n_rows, int n_ghost, const int32_t* row_ptr_h,
                    const int32_t* off_diag_offset_h, const int32_t* cols_h,
                    const double* values_h, pmgx_halo* halo, pmgx_operator** out);
/* Assemble the CSR matrix of a matrix-free Laplacian (BC rows/cols zero, diagonal 1:
 * fem::assemble_matrix + set_diagonal, src/csr.hpp:76-86); rows = owned dofs. Intended for
 * the coarse P1 level (north_star item 5). */
int pmgx_csr_from_laplacian(pmgx_operator* lap, pmgx_operator** out);
long long pmgx_csr_nnz(pmgx_operator* op);                      /* MatrixOperator::nnz :279 */
int pmgx_csr_get(pmgx_operator* op, int32_t* row_ptr_h, int32_t* cols_h, double* values_h);

/* --------------------------------------------------------- generic operator -- */
/* Operator::operator()(Vector& in, Vector& out): y = A x, incl. the zero fill and the
 * forward halo update of x overlapped with the interior cells / owned columns
 * (src/laplacian.hpp:462-482,373-460; src/csr.hpp:220-273). x's ghost block is refreshed. */
int pmgx_operator_apply(pmgx_operator* op, double* x, double* y);
/* get_diag_inverse / set_diag_inverse (src/laplacian.hpp:484-495, src/csr.hpp:205-209):
 * n_owned values. */
int pmgx_operator_get_diag_inverse(pmgx_operator* op, double* out);
int pmgx_operator_set_diag_inverse(pmgx_operator* op, const double* in);
int pmgx_operator_n_owned(pmgx_operator* op);
int pmgx_operator_n_ghost(pmgx_operator* op);
int pmgx_operator_destroy(pmgx_operator* op);

/* ---------------------------------------------------------------- Chebyshev -- */
/* acc::Chebyshev (src/chebyshev.hpp:25-91): 4th-kind, Jacobi; only eig_max is used (:51). */
int pmgx_cheb_create(pmgx_ctx* ctx, int n_owned, int n_ghost, double eig_min, double eig_max,
                     pmgx_cheb** out);
int pmgx_cheb_set_max_iterations(pmgx_cheb* s, int max_iter);
/* solve(A, x, b, verbose): resid_hist_h (max_iter+1 entries, may be NULL) receives the
 * UNPRECONDITIONED residual norms the reference prints when verbose (:59-63,85-89). */
int pmgx_cheb_solve(pmgx_cheb* s, pmgx_operator* A, double* x, const double* b,
                    double* resid_hist_h);
int pmgx_cheb_residual(pmgx_cheb* s, pmgx_operator* A, double* x, const double* b,
                       double* rnorm_h);                                   /* :37-43 */
int pmgx_cheb_destroy(pmgx_cheb* s);

/* ----------------------------------------------------------------------- CG -- */
/* acc::CGSolver (src/cg.hpp:99-222). */
int pmgx_cg_create(pmgx_ctx* ctx, int n_owned, int n_ghost, pmgx_cg** out);
int pmgx_cg_set_max_iterations(pmgx_cg* s, int max_iter);
int pmgx_cg_set_tolerance(pmgx_cg* s, double rtol);
int pmgx_cg_store_coefficients(pmgx_cg* s, int on);
/* M^-1 of the solve: NULL (default) = Jacobi, the operator's diag^-1 like src/cg.hpp:154,162,192;
 * a V-cycle handle = MultigridPreconditioner::apply from a zero initial guess (src/pmg.hpp:56) in
 * those two places -- the outer Krylov solver of SURVEY 8f-4.  The handle is borrowed; its top
 * level must have the solver's vector layout.  Use a tight coarse-solver tolerance: a truncated
 * inner Krylov solve is not a fixed linear operator. */
int pmgx_cg_set_preconditioner(pmgx_cg* s, pmgx_vcycle* M);
/* solve -> iteration count in *iters_h (the reference's return value). */
int pmgx_cg_solve(pmgx_cg* s, pmgx_operator* A, double* x, const double* b, int* iters_h);
/* alphas()/betas()/residual history as stored by the reference (:213-218); returns count. */
int pmgx_cg_num_coefficients(pmgx_cg* s);
int pmgx_cg_get_coefficients(pmgx_cg* s, double* alphas_h, double* betas_h, double* residuals_h);
/* every iteration's r.M^-1 r (also the un-stored last one) and rnorm0, for parity tests */
int pmgx_cg_get_history(pmgx_cg* s, double* rnorm0_h, double* rnorms_h, int* n_h);
/* compute_eigenvalues (:121-142): sorted Lanczos estimates, eig_h[num_coefficients]. */
int pmgx_cg_compute_eigenvalues(pmgx_cg* s, double* eig_h);
int pmgx_cg_destroy(pmgx_cg* s);

/* ------------------------------------------------------------- p-transfer -- */
/* Interpolator (src/interpolate.hpp:93-181): coarse degree Q1 -> fine degree Q2 on the same
 * cells. dofmaps are device arrays [n_cells][(P+1)^3]; lcells_h/bcells_h host lists;
 * halo_c / halo_f: forward-scatter plans of the coarse / fine vectors (may be NULL). */
int pmgx_interp_create(pmgx_ctx* ctx, int degree_coarse, int degree_fine, int n_cells,
                       const int32_t* dofmap_coarse, const int32_t* dofmap_fine,
                       int n_coarse_total, int n_fine_total,
                       const int32_t* lcells_h, int n_lcells, const int32_t* bcells_h,
                       int n_bcells, pmgx_halo* halo_c, pmgx_halo* halo_f, pmgx_interp** out);
int pmgx_interp_prolong(pmgx_interp* it, double* coarse, double* fine);   /* interpolate :185-239 */
int pmgx_interp_restrict(pmgx_interp* it, double* fine, double* coarse);  /* reverse_interpolate :245-303 */
int pmgx_interp_destroy(pmgx_interp* it);

/* ------------------------------------------------------------ coarse solver -- */
/* CoarseSolverType::solve(x, b) (src/amg.hpp:67-113; PETSc KSPCG + PCHYPRE/BoomerAMG, maxits 60, PETSc's
 * default rtol 1e-5 there): PCG on the assembled CSR operator (north_star item 5), <= max_iter
 * iterations, relative tolerance rtol on sqrt(r.M^-1 r).
 *   pmgx_coarse_create      M = Jacobi (diag^-1 of the operator)
 *   pmgx_coarse_create_amg  M = one V(nu,nu) cycle of a smoothed-aggregation hierarchy built from the
 *                           operator (host set-up pmgx_amg_setup_dist_h, device cycle: this library's CSR
 *                           SpMV + 4th-kind Chebyshev/Jacobi smoother, rank-local CSR transfers, dense
 *                           inverse of the gathered coarsest level).  COLLECTIVE with nranks > 1 (it
 *                           creates one halo plan per level).  min_coarse / max_levels <= 0: defaults. */
int pmgx_coarse_create(pmgx_ctx* ctx, pmgx_operator* A_csr, int max_iter, double rtol,
                       pmgx_coarse** out);
int pmgx_coarse_create_amg(pmgx_ctx* ctx, pmgx_operator* A_csr, int max_iter, double rtol, int nu,
                           int min_coarse, int max_levels, pmgx_coarse** out);
int pmgx_coarse_solve(pmgx_coarse* cs, double* x, const double* b, int* iters_h);
/* iterations of the most recent solve (stand-alone or inside pmgx_vcycle_apply); the host looks at
 * the residual every 8 iterations with the Jacobi preconditioner (the count is a multiple of 8 or
 * max_iter) and after every iteration with the AMG cycle */
int pmgx_coarse_last_iterations(pmgx_coarse* cs);
/* did the most recent solve reach rtol (1) or stop at max_iter (0); relative residual
 * sqrt(r.M^-1 r / r0.M^-1 r0) at the last host check.  Non-convergence is never silent. */
int pmgx_coarse_last_status(pmgx_coarse* cs, int* converged_h, double* rel_residual_h);
/* levels of the AMG hierarchy (1 for Jacobi) and, per level, out_h[0]=owned rows [1]=nnz(A_l)
 * [2]=ghosts [3]=1 if dense coarsest solve [4]=nnz(P_l); operator complexity = sum nnz / nnz(A_0) */
int pmgx_coarse_num_levels(pmgx_coarse* cs);
int pmgx_coarse_level_info(pmgx_coarse* cs, int level, long long* out_h);
/* one application of the preconditioner alone, u = M^-1 r (for tests) */
int pmgx_coarse_apply_preconditioner(pmgx_coarse* cs, const double* r, double* u);
int pmgx_coarse_destroy(pmgx_coarse* cs);

/* ------------------------------------- multilevel coarse solver: host set-up -- */
/* Set-up of the smoothed-aggregation hierarchy that pmgx_coarse_create_amg runs on the device, where
 * the reference runs PETSc CG + BoomerAMG (src/amg.hpp:33-47).  Pure host code, no GPU needed;
 * exported so that the hierarchy (A_l, P_l, lambda_max(D^-1 A_l), halo plans) can be inspected and
 * tested on the CPU.  Rows holding only their diagonal (Dirichlet rows) stay out of the hierarchy.
 * _setup_h: single rank (every column owned).  _setup_dist_h: COLLECTIVE over nranks ranks; rows are
 * this rank's owned dofs, columns >= n_owned address the ghosts of the forward-scatter plan given in
 * the pmgx_halo_create format; `allgather(user, mine, bytes, all)` must gather `bytes` bytes of every
 * rank into all[rank * bytes ...] and return 0 (the only collective the set-up uses).  Aggregates never
 * span ranks; the prolongator is smoothed with the full rows of A, so P_l has ghost columns. */
typedef int (*pmgx_allgather_fn)(void* user, const void* mine, size_t bytes, void* all);
int pmgx_amg_setup_h(int n_rows, const int32_t* row_ptr_h, const int32_t* cols_h, const double* values_h,
                     int min_coarse, int max_levels, pmgx_amg_hier** out);
int pmgx_amg_setup_dist_h(int rank, int nranks, int n_owned, int n_ghost, const int32_t* row_ptr_h,
                          const int32_t* cols_h, const double* values_h, int n_send_nbr, const int* send_ranks_h,
                          const int* send_offsets_h, const int32_t* send_idx_h, int n_recv_nbr,
                          const int* recv_ranks_h, const int* recv_offsets_h, const int32_t* recv_idx_h,
                          pmgx_allgather_fn allgather, void* user, int min_coarse, int max_levels,
                          pmgx_amg_hier** out);
/* out_h[0]=n_owned [1]=n_ghost [2]=n_send_nbr [3]=n_send [4]=n_recv_nbr [5]=n_recv
 * [6]=1 if this (coarsest) level holds rows of the dense inverse [7]=global rows of the level [8]=nnz(R_l)
 * [9]=1 if the level is REPLICATED (levels with at most PMGX_AMG_REPL_CAP = 65536 rows on the whole machine
 * live completely on every rank: n_owned = global size, no ghosts; the parent's P then addresses the
 * rank-ordered global numbering) [10]=rows of a first replicated level that this rank's restriction produces */
int pmgx_amg_level_dist_sizes(pmgx_amg_hier* h, int level, long long* out_h);
/* R_l = the rows of the global P_l^T this rank owns: (columns of P_l that are owned) x (n_owned + n_ghost)
 * CSR; with one rank R_l = P_l^T.  P_l's own columns >= its owned count address the next level's ghosts. */
int pmgx_amg_level_get_restriction(pmgx_amg_hier* h, int level, int32_t* r_ptr_h, int32_t* r_cols_h, double* r_vals_h);
/* ghost_src_h/ghost_rid_h[n_ghost]: owner rank and owner-local index of every ghost; halo plan of the
 * level; inv_rows_h[n_owned * n_global]: this rank's rows of the inverse of the gathered coarsest
 * matrix, columns ordered [owned | other ranks' entries in rank order].  Any pointer may be NULL. */
int pmgx_amg_level_dist_get(pmgx_amg_hier* h, int level, int* ghost_src_h, int32_t* ghost_rid_h, int* send_ranks_h,
                            int* send_offsets_h, int32_t* send_idx_h, int* recv_ranks_h, int* recv_offsets_h,
                            int32_t* recv_idx_h, double* inv_rows_h);
/* Host helper of the coarse solver: the CSR matrix without its stored zeros (a row's diagonal entry is kept
 * whatever its value).  pmgx_csr_from_laplacian keeps the full 27-point pattern of the P1 element matrices like
 * DOLFINx's assemble_matrix does (src/csr.hpp:66-99 copies that pattern to the device); pmgx_coarse_create_amg
 * builds its hierarchy from that pattern and runs its level-0 SpMVs and transfers on copies without the zeros.
 * out_*_h may be NULL (count only: *kept_h). */
int pmgx_csr_drop_zeros_h(int n_rows, const int32_t* ptr_h, const int32_t* cols_h, const double* vals_h,
                          int32_t* out_ptr_h, int32_t* out_cols_h, double* out_vals_h, long long* kept_h);
int pmgx_amg_num_levels(pmgx_amg_hier* h);
/* out_h[0] = (owned) rows of A_l, [1] = nnz(A_l), [2] = columns of P_l (0 on the coarsest level), [3] = nnz(P_l) */
int pmgx_amg_level_sizes(pmgx_amg_hier* h, int level, long long* out_h);
int pmgx_amg_level_get(pmgx_amg_hier* h, int level, int32_t* a_ptr_h, int32_t* a_cols_h, double* a_vals_h,
                       int32_t* p_ptr_h, int32_t* p_cols_h, double* p_vals_h, double* lmax_h);
int pmgx_amg_destroy(pmgx_amg_hier* h);

/* ------------------------------------------------------------------ V-cycle -- */
/* MultigridPreconditioner (src/pmg.hpp:22-155). Level 0 is the coarsest.  ops[n_levels],
 * smoothers[n_levels], interps[n_levels-1] (interps[i]: level i -> i+1), bc_markers[n_levels]
 * device int8 arrays (the reference takes only level 0's, :22-24; quirk Q9), coarse may be
 * NULL (then smoothers[0] is used, :106-109). */
#define PMGX_VC_DEFAULT 0
#define PMGX_VC_LITERAL_REFERENCE_BC 1  /* mask b on level 0 only, like src/pmg.hpp:100-103 */
#define PMGX_VC_DIAGNOSTICS 2           /* evaluate the reference's eager residual norms (quirk Q8) */
#define PMGX_VC_LITERAL_SEQUENCE 4      /* recompute r = b - A u after pre-smoothing with one more apply and
                                           run the smoother's A*0 on zero initial guesses, exactly like
                                           src/pmg.hpp:83-92; default reuses the smoother's residual */
int pmgx_vcycle_create(pmgx_ctx* ctx, int n_levels, pmgx_operator** ops, pmgx_cheb** smoothers,
                       pmgx_interp** interps, const int8_t** bc_markers, pmgx_coarse* coarse,
                       int flags, pmgx_vcycle** out);
/* apply(x = b, y = u): one V-cycle on the top level; rnorm_h (may be NULL) receives
 * ||b - A u|| after the cycle (the "rnorm after PMG" of :146-149). */
int pmgx_vcycle_apply(pmgx_vcycle* vc, const double* b, double* u, double* rnorm_h);
/* with PMGX_VC_DIAGNOSTICS: per-stage residual norms of the last apply, up to cap entries */
int pmgx_vcycle_get_diagnostics(pmgx_vcycle* vc, double* out_h, int cap, int* n_h);
int pmgx_vcycle_destroy(pmgx_vcycle* vc);

/* -------------------------------------------------------- box mesh (host) -- */
/* Harness-side stand-in for mesh::create_box + ghost_layer_mesh + compute_boundary_cells +
 * tp dofmaps + exterior-facet BC markers + IndexMap/Scatterer lists (examples/pmg/main.cpp:
 * 83-124,173-185,412-451; src/mesh.hpp:16-143).  Pure host code, no GPU needed.  The box
 * [0,1]^3 with nx*ny*nz cells is split into px*py*pz blocks; `rank` selects the block.
 * perturb > 0 displaces interior vertices by U(-perturb*h, perturb*h) (hash-seeded, identical
 * on all ranks). */
int pmgx_boxmesh_create(int nx, int ny, int nz, int px, int py, int pz, int rank,
                        double perturb, uint64_t seed, pmgx_boxmesh** out);
int pmgx_boxmesh_destroy(pmgx_boxmesh* m);
/* sizes: out_h[0]=n_cells (owned+ghost) [1]=n_owned_cells [2]=n_points [3]=n_lcells [4]=n_bcells */
int pmgx_boxmesh_sizes(pmgx_boxmesh* m, long long* out_h);
int pmgx_boxmesh_geometry(pmgx_boxmesh* m, double* xgeom_h, int32_t* geom_dofmap_h);
int pmgx_boxmesh_cell_lists(pmgx_boxmesh* m, int32_t* lcells_h, int32_t* bcells_h);
/* per-degree space: out_h[0]=n_owned [1]=n_ghost [2]=n_send_nbr [3]=n_send_total
 * [4]=n_recv_nbr [5]=n_recv_total [6]=n_global */
int pmgx_boxmesh_space_sizes(pmgx_boxmesh* m, int degree, long long* out_h);
/* dofmap_h[n_cells][(P+1)^3], bc_h[n_owned+n_ghost], l2g_h[n_owned+n_ghost] (canonical
 * lexicographic global id), coords_h[n_owned+n_ghost][3]; any may be NULL. */
int pmgx_boxmesh_space(pmgx_boxmesh* m, int degree, int32_t* dofmap_h, int8_t* bc_h,
                       long long* l2g_h, double* coords_h);
int pmgx_boxmesh_halo_lists(pmgx_boxmesh* m, int degree, int* send_ranks_h, int* send_offsets_h,
                            int32_t* send_idx_h, int* recv_ranks_h, int* recv_offsets_h,
                            int32_t* recv_idx_h);
/* Mesh-size fit of the drivers (examples/pmg/main.cpp:412-435): cells per direction whose
 * (n*order+1)^3 dof count is closest to ndofs_total. */
int pmgx_boxmesh_fit(long long ndofs_total, int order, int* nxyz_h);

/* ------------------------------------------- general mesh + ghost layer (host) -- */
/* Ghost-layer builder for GENERAL conforming hexahedral meshes -- arbitrary vertex numbering, cell order,
 * cell orientation and partition -- producing for `rank` the arrays the operator API takes, i.e. what
 * the reference drivers get from DOLFINx (examples/pmg/main.cpp:199-256): ghost_layer_mesh (src/mesh.hpp:
 * 16-98: every cell of another rank sharing a vertex with this rank's cells is ghosted),
 * compute_boundary_cells (:105-143), tensor-product dofmaps per degree with edge/face dofs numbered in
 * an orientation-independent frame, geometry + geometry dofmap (tp vertex order 4a+2b+c), the exterior-
 * facet Dirichlet marker and the IndexMap/Scatterer lists.  Pure host code.  The whole mesh description
 * is given on every rank: cell_vertices_h[n_cells][8] global vertex ids, cell_owner_h[n_cells] the
 * partition, coords_h[n_vertices][3].  Accessors mirror pmgx_boxmesh_*; l2g_h holds library-global dof
 * ids (vertices, then edges, faces, cell interiors); geometry's cell_gid_h[n_cells] the global cell id
 * of every local cell (owned first). */
int pmgx_ghostmesh_create(int rank, int nranks, long long n_cells, const long long* cell_vertices_h,
                          const int* cell_owner_h, long long n_vertices, const double* coords_h,
                          pmgx_ghostmesh** out);
/* The same for second-order (27-node) hexahedra: cell_nodes_h[n_cells][27] global node ids in the order of
 * PMGX_LAP_GEOM_Q2 (k = 9a + 3b + c), coords_h[n_nodes][3].  Topology -- ghosting by vertex sharing, lcells /
 * bcells, dof numbering and orientation -- uses the 8 corner nodes only; every node keeps its place in its cell's
 * tensor-product frame.  pmgx_ghostmesh_geometry then writes geom_dofmap_h[n_cells][27] (local node ids) and
 * xgeom_h over all local nodes, and pmgx_ghostmesh_space computes dof coordinates through the quadratic map.
 * Fails on node ids out of range and on a corner id repeated within a cell. */
int pmgx_ghostmesh_create_q2(int rank, int nranks, long long n_cells, const long long* cell_nodes_h,
                             const int* cell_owner_h, long long n_nodes, const double* coords_h,
                             pmgx_ghostmesh** out);
/* geometry nodes per cell of the mesh: 8 (pmgx_ghostmesh_create) or 27 (pmgx_ghostmesh_create_q2) */
int pmgx_ghostmesh_nodes_per_cell(pmgx_ghostmesh* m);
int pmgx_ghostmesh_destroy(pmgx_ghostmesh* m);
int pmgx_ghostmesh_sizes(pmgx_ghostmesh* m, long long* out_h);
int pmgx_ghostmesh_geometry(pmgx_ghostmesh* m, double* xgeom_h, int32_t* geom_dofmap_h, long long* cell_gid_h);
int pmgx_ghostmesh_cell_lists(pmgx_ghostmesh* m, int32_t* lcells_h, int32_t* bcells_h);
int pmgx_ghostmesh_space_sizes(pmgx_ghostmesh* m, int degree, long long* out_h);
int pmgx_ghostmesh_space(pmgx_ghostmesh* m, int degree, int32_t* dofmap_h, int8_t* bc_h, long long* l2g_h,
                         double* coords_h);
int pmgx_ghostmesh_halo_lists(pmgx_ghostmesh* m, int degree, int* send_ranks_h, int* send_offsets_h,
                              int32_t* send_idx_h, int* recv_ranks_h, int* recv_offsets_h, int32_t* recv_idx_h);

/* GLL-collocated load vector b_i = sum_K f(x_i) w_i |detJ_K| followed by set_bc(b = g)
 * (fem::assemble_vector + set_bc with the GLL rule, examples/pmg/main.cpp:289-295). f is
 * evaluated by the caller: fvals[n_owned+n_ghost] device array of f at the dof coordinates.
 * Result is complete on owned dofs (ghost cells contribute, like the operator). */
int pmgx_laplacian_rhs(pmgx_operator* lap, const double* fvals, double g, double* b);
/* Dirichlet marker of all exterior facets, on the device (mesh::exterior_facet_indices +
 * fem::locate_dofs_topological on the host in the reference, examples/pmg/main.cpp:173-185): marker_out[i] = 1
 * for every dof on a facet that belongs to exactly one cell, owned and ghost entries alike.  geom_dofmap
 * [n_cells][8] (tp vertex order), dofmap[n_cells][(P+1)^3] are device arrays over the owned + ghost cells of
 * a ghost-layer mesh (src/mesh.hpp:16-98); for a 27-node (PMGX_LAP_GEOM_Q2) mesh pass its corner columns
 * 0, 2, 6, 8, 18, 20, 24, 26, which are the 8-vertex map in this order; halo: the forward-scatter plan of the
 * space (NULL on one rank) --
 * facet counts are exact for owned dofs, the ghost entries are taken from their owners.  COLLECTIVE like any
 * halo update. */
int pmgx_bc_marker_exterior(pmgx_ctx* ctx, int degree, int n_cells, const int32_t* geom_dofmap,
                            const int32_t* dofmap, int n_owned, int n_ghost, pmgx_halo* halo, int8_t* marker_out);

/* fem::apply_lifting + set_bc for inhomogeneous Dirichlet data (examples/pmg/main.cpp:293-295,
 * examples/cg/main.cpp:235-237): b -= A_full g_bc on the owned rows, where A_full is this operator
 * without its Dirichlet rows/columns and g_bc = gvals at the marked dofs, 0 elsewhere; then b = gvals at
 * the marked dofs.  gvals[n_owned+n_ghost] (owned and ghost entries filled).  pmgx_laplacian_rhs calls
 * this with the constant g whenever g != 0.  Set-up phase: builds a temporary un-constrained operator. */
int pmgx_laplacian_lift(pmgx_operator* lap, const double* gvals, double* b);

#ifdef __cplusplus
}
#endif
#endif /* PMGX_H */
