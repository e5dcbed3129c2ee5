/*
 * femb200.h -- C ABI of the B200-native mechanic2d hot path.
 *
 * Drop-in boundary for ONE path of SalzmanA/fem-libraries: per-element tangent
 * integration -> CSR scatter-add -> sparse operator apply (assembled SpMV and
 * matrix-free) inside a (Jacobi-)PCG solve.  Plain pointers and sizes only: no
 * torch types, no C++ types, no exceptions cross this boundary.
 *
 * Conventions
 *  - every `d_*` pointer is DEVICE memory (sm_100a) owned by the caller unless
 *    stated otherwise; `stream` is a cudaStream_t passed as void* (NULL = legacy
 *    default stream); all calls are asynchronous with respect to the host unless
 *    they return host scalars (documented per function);
 *  - every function returns 0 on success, non-zero on error; the message of the
 *    last error of the calling thread is femb200_last_error();
 *  - global dof = 2 * node + component (blocked, bs = 2), as the reference's
 *    vector P1 space (M.cc:1107 byVDIM, F.cc:691-692);
 *  - the CSR is the dolfinx convention: rows in dof order, columns ascending and
 *    unique, structural pattern (exact zeros kept), Dirichlet rows/columns
 *    zeroed in-pattern with `diag` on the diagonal (F.cc:847-862);
 *    rowptr is int64, colidx int32, values float64.
 *
 * File:line citations are relative to the reference tree, with
 *   M.cc = MFEM/mechanic2d/asym_elasto_damage_model.cc
 *   F.cc = FEniCSx/mechanic2d/asym_elasto_damage_model.cc
 *   manual.py = FEniCSx/mechanic2d/asym_manual.py
 */
#ifndef FEMB200_H
#define FEMB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FEMB200_VERSION 100

/* element families (SURVEY.md 8c conventions) */
#define FEMB200_P1 0 /* P1 triangle, 1-point rule  (the reference: M.cc:511-512, manual.py:10,97) */
#define FEMB200_P2 1 /* P2 triangle, 3-point rule, basix dof order                                */
#define FEMB200_Q2 2 /* Q2 quadrilateral, 3x3 Gauss, tensor dof order                              */
#define FEMB200_Q1 3 /* Q1 quadrilateral, pattern only: coarse levels of the multigrid hierarchy;
                        local order (v00, v10, v01, v11); no element kernel accepts it            */

/* element-matrix layouts */
#define FEMB200_ROWMAJOR_INTERLEAVED 0 /* ufcx tabulate_tensor: A[(2a+i)*n + 2b+k]              */
#define FEMB200_COLMAJOR_BYNODES 1     /* mfem::DenseMatrix elmat(i*nd+a, k*nd+b), M.cc:647,673  */

/* tangent variants for damaged points (d > 0) */
#define FEMB200_TANGENT_CLOSED 0 /* M.cc:766-871                              */
#define FEMB200_TANGENT_AD 1     /* M.cc:100-155,752-765; admfem.hpp:672-699 */

/* operator kinds for femb200_pcg */
#define FEMB200_OP_CSR 0 /* assembled matrix of a plan         */
#define FEMB200_OP_PA 1  /* partial-assembly matrix-free apply  */

#define FEMB200_PRECOND_NONE 0
#define FEMB200_PRECOND_JACOBI 1

typedef struct femb200_plan femb200_plan; /* sparsity pattern + gather maps, owns device memory */
typedef struct femb200_pa femb200_pa;     /* partial-assembly operator (quadrature data)        */

int femb200_version(void);
const char *femb200_last_error(void);
/* host scalars: SM count and compute capability of the current device */
int femb200_device_info(int *sm_count, int *cc_major, int *cc_minor);
/* FP64 FMA throughput probe (the measured denominator of the FP64 roofline of the element kernels): one launch
 * of blocks_per_sm * SM count blocks x 256 threads x iters x 8 independent FMA chains on `stream`; the caller
 * times it.  *flops = operations of the launch (FMA = 2); d_out: *blocks_out * 256 doubles (NULL: size query). */
int femb200_fp64_probe(int blocks_per_sm, int iters, double *d_out, int64_t *blocks_out, double *flops, void *stream);

/* ------------------------------------------------------------------------
 * Element kernel.
 * Replaces: the ffcx-generated `tabulate_tensor_integral_*` of form J
 * (manual.py:102; ufcx signature, FEniCSx/mechanic2d/addprofile:6-9) called once
 * per cell by dolfinx, and mfem `damIntegrator::AssembleElementGrad`
 * (M.cc:639-916) called once per element by ParNonlinearForm::GetGradient.
 * One launch tabulates `ncells` cells; d_A is ncells x (2nd)^2, overwritten (16-byte aligned).
 *   d_x        nnodes x x_stride coordinates (x_stride 2, or 3 for xyz-padded
 *              dolfinx geometry, F.cc:213)
 *   d_xdofmap  ncells x nv geometry vertices;  d_dofmap ncells x nd scalar dofs
 *   d_E        Young modulus per cell (DG0, manual.py:22);  nu constant (manual.py:23)
 *   d_dnod     nodal damage (P1 field on the vertices, manual.py:19) or NULL (d = 0)
 *   d_u        dof vector (2*nnodes) of the current iterate or NULL
 * ------------------------------------------------------------------------ */
int femb200_tabulate_tensor_batched(int etype, int64_t ncells, double *d_A, const double *d_x, int x_stride,
                                    const int32_t *d_xdofmap, const int32_t *d_dofmap, const double *d_E, double nu,
                                    const double *d_dnod, const double *d_u, int variant, int layout, void *stream);

/* The ufcx cell-kernel signature itself (ufcx_tabulate_tensor_float64 of ffcx 0.8; FEniCSx/mechanic2d/
 * addprofile:6-9, F.cc:31-67): the symbol a dolfinx Form can hold as the kernel of the P1 form J.  Batch of one
 * with the device staging inside; A (6 x 6 row-major, interleaved dofs) is caller-owned, pre-zeroed by the
 * caller and ACCUMULATED into; host pointers; no return value (errors: A untouched, femb200_last_error()).
 *   w = [d0, d1, d2, E, u0x, u0y, u1x, u1y, u2x, u2y] (manual.py:19,22,30), c = [nu] (manual.py:23),
 *   coordinate_dofs = 3 x (x, y, z) (F.cc:213).  Parity surface; the batched entry point above is the fast one. */
void femb200_tabulate_tensor_ufcx(double *A, const double *w, const double *c, const double *coordinate_dofs,
                                  const int *entity_local_index, const uint8_t *quadrature_permutation);

/* ------------------------------------------------------------------------
 * Sparsity pattern + gather maps.
 * Replaces: dolfinx::fem::petsc::create_matrix(*J_form) (F.cc:688).
 * Builds on the device, from the cell->dof map alone: node->cell lists, the
 * node-block CSR (brp/bcol), and the per-(cell, local row) slot map used by the
 * write-once gather assembly.  Synchronises the stream (returns sizes).
 * d_dofmap / d_xdofmap must stay valid for the lifetime of the plan.
 * ------------------------------------------------------------------------ */
int femb200_plan_create(int etype, int64_t nnodes, int64_t ncells, const int32_t *d_dofmap, const int32_t *d_xdofmap,
                        void *stream, femb200_plan **out);
void femb200_plan_destroy(femb200_plan *plan);
/* host scalars: sizes of the pattern */
int femb200_plan_sizes(const femb200_plan *plan, int64_t *nnodes, int64_t *ncells, int64_t *nnz_blocks, int64_t *nnz,
                       int32_t *max_block_degree, int64_t *device_bytes);
/* device pointers owned by the plan: brp[nnodes+1] int64, bcol[nnz_blocks] int32 */
int femb200_plan_block_csr(const femb200_plan *plan, const int64_t **d_brp, const int32_t **d_bcol);
/* the same, copied into caller-allocated device arrays */
int femb200_plan_copy_block_csr(const femb200_plan *plan, int64_t *d_brp, int32_t *d_bcol, void *stream);
/* expand to the scalar CSR handed back across the boundary:
 * d_rowptr[2*nnodes+1] int64, d_colidx[nnz] int32 (caller-allocated) */
int femb200_plan_scalar_csr(const femb200_plan *plan, int64_t *d_rowptr, int32_t *d_colidx, void *stream);

/* ------------------------------------------------------------------------
 * Assembly.
 * Replaces: MatZeroEntries + dolfinx::fem::assemble_matrix(set_block_fn(A,
 * ADD_VALUES), *J_form, {bcl, bcr}) + set_diagonal(..., 1.) + MatAssembly
 * (the setJ lambda, F.cc:847-862); on the MFEM side AddDomainIntegrator /
 * SetEssentialTrueDofs / ParNonlinearForm::GetGradient (M.cc:1489-1490,1546).
 * d_values[nnz] is written once (no zero-fill needed, no atomics).
 * ------------------------------------------------------------------------ */
int femb200_assemble_matrix(const femb200_plan *plan, const double *d_x, int x_stride, const double *d_E, double nu,
                            const double *d_dnod, const double *d_u, int variant, double *d_values, void *stream);
/* assemble_matrix + (|K|_F^2, trace K) of the assembled (constrained) matrix in d_norms[0..1]: on the
 * fast path the sums are fused into the stream-out of the assembly kernel (values still in registers)
 * and corrected for the Dirichlet rows / columns, instead of a second pass over the value array */
int femb200_assemble_matrix_norms(const femb200_plan *plan, const double *d_x, int x_stride, const double *d_E, double nu,
                                  const double *d_dnod, const double *d_u, int variant, double *d_values, double *d_norms,
                                  void *stream);
/* assemble_matrix without the Dirichlet treatment (the unconstrained tangent, needed by apply_lifting) */
int femb200_assemble_matrix_nobc(const femb200_plan *plan, const double *d_x, int x_stride, const double *d_E, double nu,
                                 const double *d_dnod, const double *d_u, int variant, double *d_values, void *stream);
/* Dirichlet dofs: d_bc is a per-dof marker (uint8, 2*nnodes).  Builds the compact
 * list of constrained nodes once (F.cc:640,664 create the DirichletBC objects
 * once); pass NULL to clear.  Synchronises the stream. */
int femb200_plan_set_dirichlet(femb200_plan *plan, const uint8_t *d_bc, void *stream);
/* zero rows and columns of the marked dofs, put `diag` on their diagonal */
int femb200_apply_dirichlet(const femb200_plan *plan, double *d_values, double diag, void *stream);
/* Frobenius norm^2 and trace of the assembled matrix into d_out[2] (device) */
int femb200_matrix_norms(const femb200_plan *plan, const double *d_values, double *d_out, void *stream);

/* ------------------------------------------------------------------------
 * Residual vector (SURVEY.md 8f, rank 1).
 * Replaces: the setF lambda (F.cc:817-845) = assemble_vector(F) + apply_lifting(J,
 * bcs, u, -1) + set_bc(-1), and ParNonlinearForm::Mult ->
 * damIntegrator::AssembleElementVector + asym_stress (M.cc:559-637, 207-329).
 *   d_b[2*nnodes] = sum_e r_e, r_e = int sigma(u):eps(v) - int f.v, written once;
 *   d_u current iterate (required); d_fnod nodal body force (nnodes x 2) or NULL.
 * apply_lifting: b -= scale * K[:, bc] (g - u)_bc on the free dofs and
 *   b[bc] = scale * (g - u)[bc]  (dolfinx: scale = -1, SURVEY.md A.8), with K the
 *   UNCONSTRAINED tangent (femb200_assemble_matrix_nobc); only the node rows with a constrained
 *   column are touched (O(boundary) work); d_work: unused (may be NULL), kept in the signature.
 * ------------------------------------------------------------------------ */
int femb200_assemble_vector(const femb200_plan *plan, const double *d_x, int x_stride, const double *d_E, double nu,
                            const double *d_dnod, const double *d_u, const double *d_fnod, double *d_b, void *stream);
int femb200_apply_lifting(const femb200_plan *plan, const double *d_values_nobc, const double *d_g, const double *d_u,
                          double scale, double *d_b, double *d_work, void *stream);
/* set_bc alone (F.cc:836): b[bc] = scale * (g - u)[bc]; what the lifting reduces to once u carries the
 * boundary values (every Newton iteration after the first) */
int femb200_set_bc(const femb200_plan *plan, const double *d_g, const double *d_u, double scale, double *d_b, void *stream);
/* y += alpha x (the Newton update u <- u - du, M.cc:1546 / F.cc:894) */
int femb200_axpy(int64_t n, double alpha, const double *d_x, double *d_y, void *stream);

/* ------------------------------------------------------------------------
 * Assembled operator apply.
 * Replaces: HypreParMatrix::Mult inside mfem::CGSolver (M.cc:1502,1525-1528) /
 * PETSc MatMult inside KSP cg (F.cc:718-722).  d_values is the scalar-CSR value
 * array of femb200_assemble_matrix; the kernel walks the node-block pattern.
 * ------------------------------------------------------------------------ */
int femb200_spmv(const femb200_plan *plan, const double *d_values, const double *d_x, double *d_y, void *stream);
/* y = A x and d_dot[0] = <x, y> in the same pass (deterministic reduction) */
int femb200_spmv_dot(const femb200_plan *plan, const double *d_values, const double *d_x, double *d_y, double *d_dot,
                     void *stream);
/* y = A x on the node rows [row_lo, row_hi) only (any range: the rows a rank owns); rows outside are left
 * untouched.  d_dot (or NULL) receives <x, y> over those rows, added to its content when `accumulate`; d_flag
 * (or NULL): no-op when *d_flag != 0 (converged CG).  The first call with a range that does not start on a
 * 64-row boundary measures its tiling once (synchronises the device). */
int femb200_spmv_rows(const femb200_plan *plan, const double *d_values, const double *d_x, double *d_y, int64_t row_lo,
                      int64_t row_hi, double *d_dot, int accumulate, const double *d_flag, void *stream);
int femb200_extract_diagonal(const femb200_plan *plan, const double *d_values, double *d_diag, void *stream);
/* d_dinv[i] = 1 / d_diag[i] (Jacobi preconditioner) */
int femb200_jacobi_setup(int64_t n, const double *d_diag, double *d_dinv, void *stream);

/* ------------------------------------------------------------------------
 * (Jacobi-)PCG with mfem::CGSolver semantics (M.cc:1502,1525-1528; the PETSc
 * side is KSP cg with the same tolerances, F.cc:718-722): zero initial guess,
 * stop when <B r, r> <= max(rtol^2 <B r0, r0>, atol^2), at most maxit
 * iterations.  The reference's preconditioner B is HYPRE BoomerAMG (third
 * party, out of scope); here B = diag(A)^-1 (d_dinv) or the identity (NULL).
 *   op_kind FEMB200_OP_CSR: plan + d_values;  FEMB200_OP_PA: op = femb200_pa*
 *   n       number of dofs (2 * nnodes)
 *   d_work  3*n + 64 doubles of scratch
 * Device-resident scalars: the host polls convergence every `check_every`
 * iterations only.  `fixed_iters` > 0 runs exactly that many iterations without
 * any poll (benchmark mode).  Host scalars out: iterations, <B r, r>^(1/2),
 * converged flag.  Synchronises the stream before returning.
 * ------------------------------------------------------------------------ */
int femb200_pcg(const femb200_plan *plan, int op_kind, const void *op, const double *d_values, const double *d_b,
                double *d_x, int64_t n, double rtol, double atol, int maxit, const double *d_dinv, int check_every,
                int fixed_iters, double *d_work, int *iters, double *final_norm, int *converged, void *stream);

/* CG building blocks, used one by one by the multi-GPU driver, which all-reduces
 * the partial sums between a vector kernel and its scalar step (the analogue of
 * the MPI_Allreduce inside CGSolver / KSP).  d_scal: 16 device doubles,
 *   [0] nom [1] den [2] betanom [3] r0 [4] flag (0 run, 1 converged, 2 breakdown)
 *   [5] iterations [6] last <B r, r> [7] rtol^2 [8] atol^2
 *   [9] local <B r0, r0> [10] local <d, A d> [11] local <B r, r> [12] beta
 * Every kernel is a no-op once the flag is set. */
#define FEMB200_SC_FLAG 4
#define FEMB200_SC_ITERS 5
#define FEMB200_SC_FINAL 6
#define FEMB200_SC_RED_NOM 9
#define FEMB200_SC_RED_DEN 10
#define FEMB200_SC_RED_BETA 11
#define FEMB200_SC_COUNT 16
int femb200_dot(int64_t n, const double *d_a, const double *d_b, double *d_out, void *stream);
int femb200_cg_set_tolerances(double *d_scal, double rtol, double atol, void *stream);
/* x = 0, r = b, d = B b, scal[9] = local <d, r> */
int femb200_cg_init(int64_t n, const double *d_b, const double *d_dinv, double *d_x, double *d_r, double *d_dir,
                    double *d_scal, void *stream);
/* phase 0: after cg_init; 1: after cg_apply; 2: after cg_update_xr */
int femb200_cg_scalar_step(double *d_scal, int phase, void *stream);
/* Ad = A d, scal[10] = local <d, A d> */
int femb200_cg_apply(const femb200_plan *plan, int op_kind, const void *op, const double *d_values, const double *d_dir,
                     double *d_Ad, double *d_scal, void *stream);
/* x += alpha d, r -= alpha Ad, scal[11] = local <B r, r> */
int femb200_cg_update_xr(int64_t n, double *d_scal, const double *d_dir, const double *d_Ad, const double *d_dinv,
                         double *d_x, double *d_r, void *stream);
/* d = B r + beta d */
int femb200_cg_update_dir(int64_t n, const double *d_scal, const double *d_r, const double *d_dinv, double *d_dir,
                          void *stream);

/* d_dst[k] = d_src[d_node_idx[k]] over nodes (2 doubles each): packs the interface
 * dofs of a halo message before ncclSend (role of the dolfinx Scatterer behind
 * VecGhostUpdate(INSERT, FORWARD), F.cc:865-866) */
int femb200_gather(int64_t nnodes_out, const int32_t *d_node_idx, const double *d_src, double *d_dst, void *stream);
/* d_dst[d_idx[k]] = d_src[k] over rows of `width` doubles: refreshes the coordinates of the geometry
 * vertices only (dolfinx mesh.geometry.x holds the P1 geometry, F.cc:213) */
int femb200_scatter_rows(int64_t n, int width, const int32_t *d_idx, const double *d_src, double *d_dst, void *stream);
/* Kernel selection of a plan.  The write-once assembly and the SpMV each have a fallback kernel for
 * patterns the fast one does not cover (a node in 16 or more cells, a 64-row tile beyond the shared-memory
 * budget); these options force a path so that tests exercise the fallbacks on any mesh.  Read at launch
 * from the plan, no environment variables.
 *   "assembly_path"  0 auto | 1 visit-record kernel | 2 per-quadrature-point kernel
 *   "spmv_path"      0 auto (bulk-copy staged) | 1 direct kernel
 *   "spmv_cols"      0 auto (stencil ids: one byte per node row naming its list of column offsets in the plan's
 *                    dictionary, when the pattern has at most 64 distinct lists of at most 32 blocks; else 16-bit
 *                    column offsets from the row's node when every offset fits; else 32-bit) | 1 32-bit |
 *                    2 16-bit offsets (32-bit when an offset does not fit).  Every mode gives the same y bit for bit.
 *   "spmv_compact"   0 auto | 1 off.  Auto: on a P2 plan with compact keys (see below) the operator applies inside
 *                    femb200_pcg / femb200_dist_pcg stream a copy of the values without the vertex / opposite-edge
 *                    blocks (zero on every straight-sided cell), about a quarter fewer bytes.  The first apply of each
 *                    solve writes the copy from that solve's values and checks that every dropped block is +-0; when
 *                    one is not (curved or damaged cells, edited values) the solve streams the CSR values.  The copy
 *                    (32 B per kept block) is allocated by the first solve on the plan and shared by later ones; when
 *                    it cannot be allocated the solves stream the CSR values.  Iterates are bit-identical either way
 *                    (finite iterates).  Solves on one plan must not run concurrently.
 *   "vector_path"    residual vector: 0 two passes (element vectors per cell, then a gather per node) | 1 single-pass gather
 *   "prefetch_tiles" record prefetch distance of the assembly kernel in tiles (-1: 8 x SM count, 0: off)
 *   "stream_out"     0 auto (tensor bulk stores of the finished tile) | 1 store loop
 *   "damage_stage"   damaged reassembly: 0 auto (damage records staged per tile in shared memory once 40 % of the
 *                    cells were damaged in the previous assembly on the plan) | 1 always | 2 never */
int femb200_plan_set_option(femb200_plan *plan, const char *key, int value);
/* Reads an option back, or one of the read-only facts of the plan: "spmv_col_bits" (16 or 32: the column index
 * width the staged SpMV reads with the current options; 0: it reads stencil ids, no column indices), "spmv_stencils"
 * (the number of lists in the plan's stencil dictionary, 0: the plan has none), "spmv_compact_keys" (the number of
 * (stencil, kept blocks) keys of the compact values, 0: the plan has none), "fast_records" (1: the plan has
 * fast-path records). */
int femb200_plan_get_option(const femb200_plan *plan, const char *key, int *value);

/* ------------------------------------------------------------------------
 * Multi-GPU: one mesh partition per rank (one process per GPU).
 * Replaces: the MPI layer under the linear solve of both drivers -- the forward
 * ghost update before an operator apply (VecGhostUpdate(INSERT, FORWARD),
 * F.cc:865-866; the halo inside HypreParMatrix::Mult) and the MPI_Allreduce of
 * the CG dot products inside mfem::CGSolver / PETSc KSP cg (M.cc:1502-1528,
 * F.cc:718-722); partition = element blocks, ownership = lowest rank
 * (doc.tex:444-464, F.cc:159).
 * Local numbering: owned nodes are ONE contiguous range [own_lo, own_hi) of the
 * plan's nodes, ghost nodes around it; the rank's mesh holds every cell touching
 * an owned node, so assembly needs no communication and owned rows are complete.
 * Per neighbour k: peers[k], owned nodes [send_lo[k], send_hi[k]) to send, ghost
 * nodes [recv_lo[k], recv_hi[k]) to receive (contiguous ranges).
 * Transports (attach one or both, pick with set_transport; the last attached is
 * active):
 *   NCCL  any ncclComm_t (void*) of `world` ranks: ncclSend/ncclRecv halo,
 *         ncclAllReduce of the dot products, on the caller's stream;
 *   P2P   NVLink peer memory on one box: every rank exports its arena with
 *         p2p_export (FEMB200_DIST_BLOB_BYTES bytes), the host all-gathers the
 *         blobs (rank order) and hands them to p2p_attach.  The halo is then one
 *         kernel storing straight into the neighbours' ghost rows, the all-reduce
 *         is fused into the scalar kernel of the CG (no collective launches).
 * All ranks must issue the same sequence of dist calls.
 * ------------------------------------------------------------------------ */
typedef struct femb200_dist femb200_dist;
#define FEMB200_DIST_NCCL 1
#define FEMB200_DIST_P2P 2
#define FEMB200_DIST_BLOB_BYTES 256
int femb200_dist_create(const femb200_plan *plan, int rank, int world, int64_t own_lo, int64_t own_hi, int nneigh,
                        const int32_t *peers, const int64_t *send_lo, const int64_t *send_hi, const int64_t *recv_lo,
                        const int64_t *recv_hi, void *stream, femb200_dist **out);
void femb200_dist_destroy(femb200_dist *dist);
/* helpers for hosts without a communicator of their own: id on rank 0 (128 bytes, broadcast it), then
 * comm_create on every rank (ncclCommInitRank) */
int femb200_dist_nccl_unique_id(unsigned char *id128);
int femb200_dist_nccl_comm_create(const unsigned char *id128, int rank, int world, void **nccl_comm_out);
int femb200_dist_nccl_comm_destroy(void *nccl_comm);
int femb200_dist_attach_nccl(femb200_dist *dist, void *nccl_comm);
int femb200_dist_p2p_export(femb200_dist *dist, unsigned char *blob);
int femb200_dist_p2p_attach(femb200_dist *dist, const unsigned char *blobs_of_all_ranks);
int femb200_dist_set_transport(femb200_dist *dist, int transport);
int femb200_dist_transport(const femb200_dist *dist);
/* sum of d_vals[0..count) (count <= 3) over the ranks, in place, identical on every rank */
int femb200_dist_allreduce_sum(femb200_dist *dist, double *d_vals, int count, void *stream);
/* forward ghost update of a local dof vector (2 * plan nodes) */
int femb200_dist_halo(femb200_dist *dist, double *d_v, void *stream);
/* y[owned] = (A v)[owned] after the ghost update of v */
int femb200_dist_mult(femb200_dist *dist, const double *d_values, double *d_v, double *d_y, void *stream);
/* femb200_pcg over the ranks: d_b, d_x, d_dinv are local vectors (ghosts included, only owned entries are
 * read / written); `use_graph` replays one captured CUDA graph per iteration; host scalars are identical on
 * every rank; synchronises the stream.  world = 1 needs no transport. */
int femb200_dist_pcg(femb200_dist *dist, int op_kind, const void *op, const double *d_values, const double *d_b,
                     double *d_x, double rtol, double atol, int maxit, const double *d_dinv, int check_every,
                     int fixed_iters, int use_graph, int *iters, double *final_norm, int *converged, void *stream);
/* work vectors of the communicator after a solve (device pointers, local length): recurrence residual r,
 * search direction, A d, and the 16 CG scalars */
int femb200_dist_vectors(femb200_dist *dist, double **d_r, double **d_dir, double **d_z, double **d_scal);

/* ------------------------------------------------------------------------
 * Partial assembly (matrix-free).
 * Role of mfem BilinearFormIntegrator::AssemblePA / AddMultPA (not exercised by
 * the reference, discussed at doc.tex:1445-1449): per-cell data once
 * (pa_create = AssemblePA), then y = A x by element-local sum-factorised
 * contractions (pa_apply = AddMultPA into a zeroed y).
 * d_dofmap must stay valid for the lifetime of the operator.
 * ------------------------------------------------------------------------ */
int femb200_pa_create(int etype, int64_t nnodes, int64_t ncells, const int32_t *d_dofmap, const int32_t *d_xdofmap,
                      const double *d_x, int x_stride, const double *d_E, double nu, void *stream, femb200_pa **out);
void femb200_pa_destroy(femb200_pa *pa);
/* per-dof marker (uint8, 2*nnodes) or NULL to clear; synchronises the stream */
int femb200_pa_set_dirichlet(femb200_pa *pa, const uint8_t *d_bc, double diag, void *stream);
/* y = A x (overwrites y) */
int femb200_pa_apply(const femb200_pa *pa, const double *d_x, double *d_y, void *stream);
int femb200_pa_diagonal(const femb200_pa *pa, double *d_diag, void *stream);

/* ------------------------------------------------------------------------
 * Field operators either side of the hot path (SURVEY.md 8f ranks 3-4).
 * smooth_damage: the reference's damage-field smoothing over the vertex graph
 * (M.cc:1258-1315; F.py:160-199): niter double sweeps d_l = max(sum over edge
 * neighbours / degree, d_l), the first sweep of a pair only where d_l < threshold
 * (0.01 in the reference).  `plan` is the P1 plan of the triangulation (its block
 * pattern is the edge graph plus the diagonal); d_d [nnodes] in/out, d_work
 * [nnodes] scratch.  The reference runs niter = 8 * (max_refine + 1).
 * cell_strain_stress: DG0 output fields (strainTensor / stressTensor,
 * M.cc:333-430,1551-1563; F.cc:909-942): symmetric gradient of u and asym_stress
 * at the cell centroid, three doubles (xx, xy, yy) per cell; d_strain or d_stress
 * may be NULL; d_dnod (nodal damage on the geometry vertices) may be NULL (d = 0).
 * ------------------------------------------------------------------------ */
int femb200_smooth_damage(const femb200_plan *plan, double *d_d, double *d_work, int niter, double threshold,
                          void *stream);
int femb200_cell_strain_stress(int etype, int64_t ncells, const int32_t *d_xdofmap, const int32_t *d_dofmap,
                               const double *d_x, int x_stride, const double *d_E, double nu, const double *d_dnod,
                               const double *d_u, double *d_strain, double *d_stress, void *stream);

/* ------------------------------------------------------------------------
 * Geometric multigrid preconditioner (single GPU).
 * Levels 0 (the fine operator, Dirichlet applied through its marker) .. L (coarsest).  Level 0 is an assembled
 * plan (FEMB200_OP_CSR: P1, P2 or Q2) or a matrix-free operator (FEMB200_OP_PA: P2 or Q2); levels 1..L are P1
 * plans (map width 2) or Q1 plans (map width 4).
 * Transfer map of level l, per level-l node, `width` int32 level-(l+1) node ids:
 *   width 2  (a, b): a == b a coincident node (weight 1), else the midpoint of the coarse edge (a, b) (1/2 each);
 *   width 4  (a, a, a, a) a coincident node, (a, b, a, b) the midpoint of edge (a, b), (v00, v10, v01, v11) the
 *            centre of a coarse quad; each distinct entry weighs 1 / (number of distinct entries).
 * Entry k and its partner (width - 1 - k) name the coarse block slots a fine node stands for: its diagonal block,
 * its edge, or the two diagonals of its quad.  Both components alike.  P has zero rows for constrained fine dofs
 * and zero columns for constrained coarse dofs (the levels' markers).
 *   mg_create_op    borrows the fine operator and the plans (they must outlive the handle); sets the coarse plans'
 *                   Dirichlet markers from d_coarse_bc[l] (uint8 per dof, NULL: none); validates that the maps
 *                   are nested (every pair in the coarse pattern, every coarse slot hit by exactly one fine node);
 *                   Chebyshev smoother of `degree` on D^-1 A over [lo_frac lambda, lambda].  Synchronises.
 *                   OP_CSR: fine_op is the fine plan.  OP_PA: fine_op is a femb200_pa (its own Dirichlet marker
 *                   and diagonal, read at every call); the first step must be a p-coarsening (P2 -> P1, Q2 -> Q1):
 *                   the map row of every node of fine cell k names the vertices of coarse cell k the element
 *                   interpolation weights it on (checked on the device).  Destroying the operator invalidates the
 *                   handle: create a new one on the new operator.
 *   mg_create       = mg_create_op(FEMB200_OP_CSR, fine, ..., width 2, ...)
 *   mg_sizes        host: L, and per level 0..L dofs, nnz (0 for a matrix-free level 0), lambda (1.1 x 15-step
 *                   power iteration, after setup), device bytes of the handle
 *   mg_galerkin     A_{level+1} = P^T A_level P (gather kernel, write-once) + unit Dirichlet diagonal;
 *                   level 0 reads d_fine_values (kept by the handle: it must stay valid).  Matrix-free level 0:
 *                   d_fine_values must be NULL; sum over the cells of P_e^T K_e P_e from the operator's own
 *                   geometry and quadrature, gathered through the coarse plan's visit records (no fine matrix;
 *                   a per-cell scratch of (2 nv)^2 doubles is allocated on `stream` for the call only)
 *   mg_setup        the numeric phase: every mg_galerkin, D^-1 and lambda per level.  Synchronises.  Re-run
 *                   after every reassembly of the fine values, then hand in a new coarse inverse.  d_fine_values:
 *                   NULL for a matrix-free level 0.
 *   mg_level_values copy of the CSR values of level 1..L (the pattern of that level's plan)
 *   mg_coarse_matrix / mg_set_coarse_inverse: dense row-major image of A_L (n_L^2 doubles), and its inverse
 *                   (copied into the handle; the V-cycle applies it with a GEMV kernel)
 *   mg_restrict     d_bc = P^T (d_b - d_t) from level to level + 1 (d_t = A x, or NULL for x = 0)
 *   mg_prolong      d_x += P d_xc from level + 1 to level
 *   mg_vcycle       z = B r (z != r): one symmetric V(degree, degree) cycle with an exact coarse solve
 *   pcg_mg          femb200_pcg with B = mg_vcycle (mfem::CGSolver semantics, nom = <B r, r>); d_work: 4 n + 64
 *                   doubles; host poll every check_every iterations (<= 0: every one).  Synchronises.
 * ------------------------------------------------------------------------ */
typedef struct femb200_mg femb200_mg;
int femb200_mg_create(const femb200_plan *fine, int nlevels, femb200_plan *const *coarse_plans,
                      const int32_t *const *d_maps, const uint8_t *const *d_coarse_bc, int degree, double lo_frac,
                      void *stream, femb200_mg **out);
int femb200_mg_create_op(int op_kind, const void *fine_op, int nlevels, femb200_plan *const *coarse_plans,
                         const int32_t *const *d_maps, int map_width, const uint8_t *const *d_coarse_bc, int degree,
                         double lo_frac, void *stream, femb200_mg **out);
void femb200_mg_destroy(femb200_mg *mg);
int femb200_mg_sizes(const femb200_mg *mg, int *nlevels, int64_t *ndofs, int64_t *nnz, double *lambda,
                     int64_t *device_bytes);
int femb200_mg_galerkin(femb200_mg *mg, const double *d_fine_values, int level, void *stream);
int femb200_mg_setup(femb200_mg *mg, const double *d_fine_values, void *stream);
int femb200_mg_level_values(const femb200_mg *mg, int level, double *d_out, void *stream);
int femb200_mg_coarse_matrix(const femb200_mg *mg, double *d_dense, void *stream);
int femb200_mg_set_coarse_inverse(femb200_mg *mg, const double *d_inv, void *stream);
int femb200_mg_restrict(const femb200_mg *mg, int level, const double *d_b, const double *d_t, double *d_bc, void *stream);
int femb200_mg_prolong(const femb200_mg *mg, int level, const double *d_xc, double *d_x, void *stream);
int femb200_mg_vcycle(femb200_mg *mg, const double *d_r, double *d_z, void *stream);
/* the same V-cycle with a CUDA event after every launch; ms[(L + 1) * 5] (host) receives per level the milliseconds
 * of its SpMVs, Chebyshev vector passes, restriction, prolongation and coarse GEMV (event to event, launch gaps
 * included).  Synchronises. */
int femb200_mg_vcycle_timed(femb200_mg *mg, const double *d_r, double *d_z, double *ms, void *stream);
int femb200_pcg_mg(femb200_mg *mg, const double *d_b, double *d_x, double rtol, double atol, int maxit, int check_every,
                   double *d_work, int *iters, double *final_norm, int *converged, void *stream);

/* ------------------------------------------------------------------------
 * The same entry points under the names SURVEY.md 8b gives the boundary.
 *   create_pattern       = plan_create        (dolfinx create_matrix, F.cc:688)
 *   element_grad_batched = tabulate_tensor_batched in the MFEM layout: elmat column-major,
 *                          dofs byNODES (damIntegrator::AssembleElementGrad, M.cc:639,673)
 *   assemble_pa          = pa_create          (BilinearFormIntegrator::AssemblePA)
 *   add_mult_pa          : y += A x           (AddMultPA; accumulated inside the apply kernel, d_work unused: may be NULL)
 *   cg                   = pcg with its own scratch and Jacobi set-up (CGSolver::Mult /
 *                          KSPSolve; precond FEMB200_PRECOND_NONE | _JACOBI); synchronises
 * ------------------------------------------------------------------------ */
int femb200_create_pattern(int etype, int64_t nnodes, int64_t ncells, const int32_t *d_dofmap, const int32_t *d_xdofmap,
                           void *stream, femb200_plan **out);
int femb200_element_grad_batched(int etype, int64_t ncells, double *d_elmat, const double *d_x, int x_stride,
                                 const int32_t *d_xdofmap, const int32_t *d_dofmap, const double *d_E, double nu,
                                 const double *d_dnod, const double *d_u, int variant, void *stream);
int femb200_assemble_pa(int etype, int64_t nnodes, int64_t ncells, const int32_t *d_dofmap, const int32_t *d_xdofmap,
                        const double *d_x, int x_stride, const double *d_E, double nu, void *stream, femb200_pa **out);
int femb200_add_mult_pa(const femb200_pa *pa, int64_t ndofs, const double *d_x, double *d_y, double *d_work, void *stream);
int femb200_cg(const femb200_plan *plan, int op_kind, const void *op, const double *d_values, const double *d_b,
               double *d_x, int64_t n, double rtol, double atol, int maxit, int precond, int *iters, double *final_res,
               int *converged, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* FEMB200_H */
