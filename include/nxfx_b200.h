/*
 * nxfx_b200.h -- C ABI of the B200-native hydraulic-network assemble+solve path.
 *
 * This is the drop-in boundary for the hot path of scientificcomputing/networks_fenicsx
 * (NetworkMesh -> HydraulicNetworkAssembler.assemble() -> Solver.solve()).  The reference has no
 * native code of its own: at these call sites it enters DOLFINx C++ / FFCx kernels / PETSc / MUMPS.
 * Each entry point below names the reference call site(s) (file:line under
 * src/networks_fenicsx/) whose native work it replaces.
 *
 * Conventions
 *   - every function returns 0 on success and a negative nxfx_status on failure; the message is
 *     available from nxfx_last_error(ctx).  Nothing falls back to the CPU.
 *   - pointers suffixed _h are HOST pointers, _d are DEVICE pointers on the ctx's GPU.
 *   - the caller owns every buffer it passes in; buffers returned by nxfx_csr_device /
 *     nxfx_mesh_geometry_device are borrowed views owned by the ctx (valid until the next
 *     nxfx_set_network / nxfx_destroy).
 *   - one ctx per GPU per process; a ctx is not thread-safe; all work is enqueued on the ctx's
 *     stream (nxfx_set_stream, default: the legacy default stream) and is asynchronous unless
 *     stated otherwise.
 *   - all reals are IEEE binary64, all indices int32_t (DOLFINx local index width).
 *
 * Global unknown order: [flux slots (colour blocks 0..C-1), pressure (one per cell), multipliers
 * (one per bifurcation)] -- assembly.py:318-321, solver.py:122-125.
 */
#ifndef NXFX_B200_H
#define NXFX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NXFX_ABI_VERSION 2

typedef struct nxfx_ctx nxfx_ctx;

typedef enum {
  NXFX_OK = 0,
  NXFX_ERR_INVALID = -1,       /* bad argument / call order */
  NXFX_ERR_CUDA = -2,          /* CUDA runtime error */
  NXFX_ERR_NOT_CONVERGED = -3, /* mirrors ksp_error_if_not_converged=True, solver.py:64 */
  NXFX_ERR_NCCL = -4,
  NXFX_ERR_UNSUPPORTED = -5,
  NXFX_ERR_COMM = -6           /* peer exchange: a rank could not be mapped / did not arrive */
} nxfx_status;

/* ---- context ------------------------------------------------------------------------------ */
int nxfx_abi_version(void);
int nxfx_create(nxfx_ctx** out, int device);
int nxfx_destroy(nxfx_ctx* ctx);
const char* nxfx_last_error(const nxfx_ctx* ctx);
int nxfx_set_stream(nxfx_ctx* ctx, void* cuda_stream); /* cudaStream_t */
int nxfx_sync(nxfx_ctx* ctx);                          /* cudaStreamSynchronize */
/* number of kernels this library has launched on ctx since creation (bench.py "gpu_launches") */
int64_t nxfx_launch_count(const nxfx_ctx* ctx);

/* device / pinned-host memory helpers (PETSc Vec / Mat storage stand-ins) */
int nxfx_malloc(nxfx_ctx* ctx, size_t bytes, void** out_d);
int nxfx_free(nxfx_ctx* ctx, void* ptr_d);
int nxfx_host_alloc(nxfx_ctx* ctx, size_t bytes, void** out_h); /* pinned */
int nxfx_host_free(nxfx_ctx* ctx, void* ptr_h);
int nxfx_memcpy_h2d(nxfx_ctx* ctx, void* dst_d, const void* src_h, size_t bytes); /* async */
int nxfx_memcpy_d2h(nxfx_ctx* ctx, void* dst_h, const void* src_d, size_t bytes); /* async */
int nxfx_memcpy_d2d(nxfx_ctx* ctx, void* dst_d, const void* src_d, size_t bytes); /* async */
int nxfx_memset(nxfx_ctx* ctx, void* dst_d, int byte, size_t bytes);              /* async */
/* CUDA-event timer on the ctx stream (bench.py) */
int nxfx_timer_start(nxfx_ctx* ctx);
int nxfx_timer_stop(nxfx_ctx* ctx, double* elapsed_ms); /* synchronises */

/* ---- (1) graph -> mesh -------------------------------------------------------------------- *
 * Replaces the mesh-array construction and dolfinx.mesh.create_mesh: mesh.py:270-324, 341-348.
 * Inputs are the host-side graph tables built by NetworkMesh (mesh.py:175-225):
 *   node_pos_h [n_nodes*gdim]  node coordinates in graph.nodes() order
 *   edge_u_h/edge_v_h [n_edges] endpoints in graph.edges() order (cells run u -> v)
 *   edge_slot_h [n_edges]       flux slot of the edge: its N+1 flux dofs are rows
 *                               slot*(N+1) .. slot*(N+1)+N  (slot = colour-block offset + rank)
 *   node_lm_h [n_nodes]         multiplier index of the node (position in bifurcation_values)
 *                               or -1 for non-bifurcation nodes
 *   bif_ptr_h [n_bif+1], bif_inc_h [I]  incidences of each bifurcation, sorted by flux slot:
 *                               entry = 2*edge + 1 for an in-edge (edge ends at the node),
 *                               2*edge for an out-edge.
 * Builds on the device: vertex records x[n_vertices][4] = {x, y, z, p_bc} (graph nodes first, then
 * the N-1 interior points of every edge, start*(1-w)+end*w, bit-identical to the reference
 * formula); one 32-byte record per vertex so that a cell's geometry and boundary data arrive in
 * one sector each.                                                                                 */
int nxfx_set_network(nxfx_ctx* ctx, int32_t n_nodes, int32_t n_edges, int32_t gdim,
                     int32_t cells_per_edge, const double* node_pos_h, const int32_t* edge_u_h,
                     const int32_t* edge_v_h, const int32_t* edge_slot_h, const int32_t* node_lm_h,
                     int32_t n_bif, const int32_t* bif_ptr_h, const int32_t* bif_inc_h);
/* re-upload node positions (same topology) and regenerate the vertex coordinates */
int nxfx_update_node_positions(nxfx_ctx* ctx, const double* node_pos_h);
int nxfx_get_sizes(const nxfx_ctx* ctx, int64_t* n_vertices, int64_t* n_cells, int64_t* n_dofs,
                   int64_t* nnz);
int nxfx_mesh_geometry_device(nxfx_ctx* ctx, const double** x_d); /* [n_vertices][4]: x, y, z, p_bc */

/* ---- (2) symbolic phase ------------------------------------------------------------------- *
 * Replaces dolfinx.fem.petsc.create_matrix (sparsity pattern + preallocation): solver.py:43,
 * assembly.py:354.  Builds the CSR pattern (rowptr, sorted colidx) on the device, including the
 * explicit zeros DOLFINx stores in the multiplier blocks.                                         */
int nxfx_symbolic(nxfx_ctx* ctx);
int nxfx_csr_device(nxfx_ctx* ctx, const int32_t** rowptr_d, const int32_t** colidx_d,
                    double** values_d); /* values of the BOUND matrix */

/* Matrices on the ctx's pattern.  The reference hands out independent PETSc Mats: Solver.__init__
 * (solver.py:43) creates one, every assembler.assemble() without A creates another
 * (assembly.py:354).  A matrix owns its CSR values and the per-cell R*h the network-Schur
 * factorisation is built from; it records how many assemblies were accumulated into it
 * (ADD_VALUES without zeroEntries).  The BOUND matrix is the target of nxfx_assemble and the
 * operator of nxfx_spmv / nxfx_residual / nxfx_pc_* / nxfx_solve.  The symbolic phase creates and
 * binds matrix 0; a new pattern (nxfx_symbolic / nxfx_set_generic_system / nxfx_set_network)
 * destroys every matrix of the old one.  Binding another matrix invalidates the factorisation.   */
int nxfx_matrix_create(nxfx_ctx* ctx, int64_t* mat_id); /* zeroed values */
int nxfx_matrix_destroy(nxfx_ctx* ctx, int64_t mat_id);
int nxfx_matrix_bind(nxfx_ctx* ctx, int64_t mat_id);
int nxfx_matrix_zero(nxfx_ctx* ctx);                    /* MatZeroEntries on the bound matrix */
int nxfx_matrix_info(nxfx_ctx* ctx, int64_t* mat_id, int32_t* assembled, int32_t* acc_count);
/* Pattern-only entries.  With flux degree 1 / pressure degree 0 the pressure rows ({-1, +1}) and the
 * multiplier rows ((0, +1) / (-1, 0)) of the matrix depend on the pattern alone.  After a non-accumulating
 * lhs nxfx_assemble the bound matrix remembers that its values hold them, and the next non-accumulating
 * assembly writes only the flux rows (and b).  nxfx_matrix_zero, an accumulating assembly and a new pattern
 * forget it.  A caller that writes the values itself through the pointer of nxfx_csr_device (or any copy of
 * it) must bind that matrix and call nxfx_matrix_touch after the write and before the next nxfx_assemble --
 * as PETSc's MatSeqAIJGetArray is followed by MatSeqAIJRestoreArray.  nxfx_matrix_static_valid reports the
 * state (1: the next overwrite skips those rows).                                                 */
int nxfx_matrix_touch(nxfx_ctx* ctx);
int nxfx_matrix_static_valid(nxfx_ctx* ctx, int32_t* valid);

/* ---- (3) numeric assembly ----------------------------------------------------------------- *
 * Replaces fem.petsc.assemble_matrix + A.assemble() + assemble_vector + ghost update:
 * assembly.py:352-367 (forms: assembly.py:253-277).
 *   nxfx_set_boundary_pressure  p_bc interpolated into P1 on the parent mesh (assembly.py:225-234),
 *                               pbc_vertex_d [n_vertices]; stored in the vertex records
 *   R_cell_d / f_cell_d [n_cells] per-cell coefficients, or NULL to use R_const / f_const
 *                               (defaults R=1, f=0: assembly.py:201-205)
 *   lhs / rhs                   assemble_lhs / assemble_rhs flags (assembly.py:333-334)
 *   accumulate                  0: overwrite (the matrix/vector was zeroed: solver.py:97-100);
 *                               1: add to the existing entries (PETSc ADD_VALUES semantics)
 *   b_d [n_dofs]                right-hand side (written when rhs != 0)
 * Matrix values go to the bound matrix (nxfx_matrix_bind; default: matrix 0).  The per-cell R*h
 * that the solver's factorisation uses is written / accumulated together with the values (lhs
 * only), so the factorisation always belongs to the matrix as it stands: a second accumulated
 * assembly, or an rhs-only re-assembly with a different R, cannot put the two out of step.        */
int nxfx_set_boundary_pressure(nxfx_ctx* ctx, const double* pbc_vertex_d);
int nxfx_assemble(nxfx_ctx* ctx, const double* R_cell_d, double R_const, const double* f_cell_d,
                  double f_const, int lhs, int rhs, int accumulate, double* b_d);

/* ---- (4) solve ---------------------------------------------------------------------------- *
 * Replaces KSP/PC/MUMPS: solver.py:41,51,58-73,127.                                              */
typedef enum { NXFX_KSP_PREONLY = 0, NXFX_KSP_FGMRES = 1 } nxfx_ksp_type;
typedef enum {
  NXFX_PC_NETWORK_SCHUR = 0, /* exact Schur complement on the multipliers (tree elimination) */
  NXFX_PC_NONE = 1,
  NXFX_PC_JACOBI_FLUX = 2    /* diag(M) on fluxes, identity elsewhere */
} nxfx_pc_type;

typedef struct {
  int32_t ksp_type;     /* nxfx_ksp_type */
  int32_t pc_type;      /* nxfx_pc_type */
  double rtol;          /* relative residual tolerance ||b-Ax|| / ||b|| */
  double atol;
  int32_t max_it;
  int32_t restart;      /* FGMRES restart length */
  int32_t refine_steps; /* PREONLY: iterative-refinement steps after the first apply */
  int32_t error_if_not_converged;
  int32_t final_residual; /* PREONLY: also evaluate the true residual of the final iterate */
  int32_t reserved;
  double refine_rtol;     /* PREONLY: refinement stops as soon as ||b - A x|| <= refine_rtol ||b||;
                             0 = always apply refine_steps corrections */
} nxfx_solve_opts;

#define NXFX_HISTORY_LEN 128
typedef struct {
  int32_t iterations;
  int32_t converged;
  double rhs_norm;
  double residual_norm;               /* final true residual ||b - A x||_2 */
  int32_t history_len;
  double history[NXFX_HISTORY_LEN];   /* residual norms (ksp_monitor) */
} nxfx_solve_info;

/* Elimination schedule of the bifurcation tree, built on the host by the Solver from the graph:
 *   t_of_bif [n_bif]      position of each multiplier in schedule order
 *   t_parent [n_bif]      parent (schedule index) or -1
 *   t_pedge  [n_bif]      graph edge joining the node to its parent or -1
 *   t_cptr [n_bif+1], t_cidx [..]  children lists (schedule indices)
 *   n_chunks, chunk_lptr [n_chunks+1]  chunks = subtrees solved by one thread block; the LAST
 *                         chunk is the top of the forest.  Levels of chunk c are
 *                         lvl_ptr[chunk_lptr[c] .. chunk_lptr[c+1]] (ranges of schedule indices,
 *                         shallowest level first).
 *   n_chords, chord_edge  graph edges between bifurcations that are not in the spanning forest
 *                         (cyclic graphs; their conductance stays on the diagonals only).          */
int nxfx_set_tree_schedule(nxfx_ctx* ctx, const int32_t* t_of_bif_h, const int32_t* t_parent_h,
                           const int32_t* t_pedge_h, const int32_t* t_cptr_h,
                           const int32_t* t_cidx_h, int32_t n_chunks, const int32_t* chunk_lptr_h,
                           int32_t n_lvl_ptr, const int32_t* lvl_ptr_h, int32_t n_chords,
                           const int32_t* chord_edge_h);
int nxfx_pc_setup(nxfx_ctx* ctx);                                    /* numeric factorisation */
int nxfx_pc_apply(nxfx_ctx* ctx, const double* r_d, double* z_d);    /* z = P^{-1} r */
int nxfx_spmv(nxfx_ctx* ctx, const double* x_d, double* y_d);        /* y = A x */
int nxfx_residual(nxfx_ctx* ctx, const double* b_d, const double* x_d, double* r_d,
                  double* norm2_h);  /* r = b - A x; *norm2_h = ||r||_2^2 (synchronises) */
int nxfx_solve(nxfx_ctx* ctx, const double* b_d, double* x_d, const nxfx_solve_opts* opts,
               nxfx_solve_info* info); /* synchronises before returning */

/* Solution mirror: replaces the device->host side of dolfinx.fem.petsc.assign (solver.py:134) for callers
 * that want the solution in host memory.  With a pinned x_h (nxfx_host_alloc, n_dofs doubles) set,
 * nxfx_solve copies x into it on a side stream as soon as the (last) back-substitution is enqueued --
 * the download overlaps the residual check -- and returns after both have finished.  NULL disables.   */
int nxfx_set_solution_mirror(nxfx_ctx* ctx, double* x_h);

/* ---- (5) end-to-end host-buffer call (bench.py "e2e") -------------------------------------- *
 * One assemble+solve step with HOST inputs and outputs: uploads node positions and p_bc vertex
 * values, regenerates the vertices, assembles, solves, downloads x.  All host pointers should be
 * pinned (nxfx_host_alloc) for full PCIe bandwidth.                                               */
int nxfx_assemble_solve_host(nxfx_ctx* ctx, const double* node_pos_h, const double* pbc_vertex_h,
                             double R_const, double f_const, const nxfx_solve_opts* opts,
                             double* x_h, nxfx_solve_info* info);

/* ---- (7) table-driven assembly for higher-order elements ------------------------------------- *
 * flux_degree / pressure_degree other than (1, 0): assembly.py:127-146 (spaces) + :253-277 (forms)
 * with P_fd flux and continuous P_pd pressure.  The pattern and the contribution lists come from
 * the host (networks_fenicsx_b200/generic.py):
 *   rowptr_h [n_dofs+1], colidx_h [nnz]   CSR pattern (explicit zeros included)
 *   src_id_h [nnz][2]   cell | (1<<30 if the value is coef * R*h of the cell), or -1
 *   src_coef_h [nnz][2] reference-element coefficient (M_ref, +-B_ref, +-trace)
 *   bsrc_ptr_h [n_dofs+1], bsrc_id_h, bsrc_coef_h   right-hand-side sources per row:
 *                       cell -> coef * f*h, vertex | (1<<30) -> coef * p_bc(vertex)
 * nxfx_assemble_generic has the semantics of nxfx_assemble.  nxfx_spmv / nxfx_solve (FGMRES with
 * pc none|jacobi) work on the resulting matrix.                                                    */
int nxfx_set_generic_system(nxfx_ctx* ctx, int32_t n_dofs, int32_t n_flux_rows, int32_t nnz,
                            const int32_t* rowptr_h, const int32_t* colidx_h, const int32_t* src_id_h,
                            const double* src_coef_h, const int32_t* bsrc_ptr_h,
                            const int32_t* bsrc_id_h, const double* bsrc_coef_h);
int nxfx_assemble_generic(nxfx_ctx* ctx, const double* R_cell_d, double R_const,
                          const double* f_cell_d, double f_const, int lhs, int rhs, int accumulate,
                          double* b_d);

/* Exact condensation (direct solve) for the table-driven path: what PCLU / MUMPS does for any polynomial
 * degree in the reference (assembly.py:121-146, solver.py:58-65).  Per graph edge the unknowns that live on
 * the edge only (flux dofs, pressure dofs inside it, pressure of a boundary node at its end) are eliminated
 * by a banded LU with partial pivoting; the bifurcation system with 2 x 2 blocks {P_b, lam_b} is eliminated
 * over the schedule of nxfx_set_tree_schedule.  After this call pc_type NXFX_PC_NETWORK_SCHUR works on
 * the generic path (exact on trees, spanning-forest approximation inside FGMRES on graphs with cycles).
 * The tables list the entries of K_e, C_e, D_e per edge type t = (u is a bifurcation) + 2 (v is a
 * bifurcation), concatenated over the 4 types with [5]-sized offset arrays (networks_fenicsx_b200/condense.py):
 *   type_n[4]                      local unknowns per type (<= n_max)
 *   loc_kind / loc_off             global dof of a local unknown: 0 flux slot*flux_dofs_per_edge+off,
 *                                  1 pcell_base+e*pcell_stride+off, 2 interior pressure vertex off of the edge,
 *                                  3 / 4 pressure of node u / v
 *   k_row, k_col, k_cell, k_coef   K_e entries: coef * (R h of cell k_cell of the edge | 1 if k_cell < 0);
 *                                  |row - col| <= kl
 *   c_row, c_slot, c_coef          C_e (local row, nodal slot 0 P_u, 1 lam_u, 2 P_v, 3 lam_v)
 *   d_slot, d_col, d_coef          D_e (nodal row slot, local column)
 *   bif_node_h [n_bif]             graph node of every bifurcation                                        */
int nxfx_set_condensation(nxfx_ctx* ctx, int32_t continuous_pressure, int32_t flux_dofs_per_edge,
                          int32_t n_max, int32_t kl, int32_t pcell_base, int32_t pcell_stride,
                          const int32_t* type_n_h, const int32_t* loc_ptr_h, const int32_t* loc_kind_h,
                          const int32_t* loc_off_h, const int32_t* k_ptr_h, const int32_t* k_row_h,
                          const int32_t* k_col_h, const int32_t* k_cell_h, const double* k_coef_h,
                          const int32_t* c_ptr_h, const int32_t* c_row_h, const int32_t* c_slot_h,
                          const double* c_coef_h, const int32_t* d_ptr_h, const int32_t* d_slot_h,
                          const int32_t* d_col_h, const double* d_coef_h, const int32_t* bif_node_h);

/* ---- (6) multi-GPU: one rank's part of a partitioned network ------------------------------------ *
 * Replaces what MPI does inside DOLFINx/PETSc/MUMPS at assembly.py:355-367 and solver.py:127-132
 * (stash exchange, ghost updates, distributed LU).  The ctx holds one rank's sub-network in which
 * the multipliers of the SHARED bifurcations -- the nodes of the elimination tree whose subtree spans
 * several ranks: world-1 of them for a balanced binary tree -- are REPLICATED (see
 * networks_fenicsx_b200/distributed.py); the rest of the top of the tree is private to one rank.
 * Every quantity that couples ranks is additive.  Either the library exchanges it itself (nxfx_comm_*
 * below: in-kernel, over NVLink), or the caller all-reduces (SUM) the small buffers between the
 * begin/end halves with its own communicator (torch.distributed / NCCL):
 *   shared_lm_h [n_shared]   local multiplier indices of the shared multipliers, in an order that is
 *                            the same on every rank (ascending global node id); they must belong to
 *                            the LAST chunk of the schedule
 *   lam_weight_h [n_bif]     1 where this rank counts the multiplier row (norms, -r_lambda), else 0
 *   buf_d                    caller-owned device buffer, sections sized by nxfx_exchange_sizes
 *   nxfx_pc_setup_begin  -> buf = [partial pivots | link conductances] of the shared nodes (2 n_shared)
 *   nxfx_pc_setup_end    <- all-reduced buf: factorises the top chunk
 *   nxfx_pc_apply_begin  -> buf[0:n_shared] = partial right-hand side of the shared nodes (may be called
 *                        right after nxfx_pc_setup_begin with a second buffer: setup and first
 *                        application then share ONE all-reduce, followed by _setup_end, _apply_end)
 *   nxfx_pc_apply_end    <- all-reduced buf: top solve, back-substitution; z = or += P^{-1} r
 *   nxfx_pc_setup_apply_begin / _end  the recommended form of that fused sequence: buf = 3*n_shared
 *                        doubles [partial pivots | link conductances | partial right-hand side],
 *                        one all-reduce in between, z = P^{-1} r.  With one cell per edge the
 *                        bottom chunks are factorised WHILE their right-hand sides are eliminated.
 *   nxfx_residual_partial  r = b - A x (local part) and buf = [shared rows of r | partial ||r||^2
 *                        over the non-shared owned rows | owned ||b||^2]  (n_shared + 2 doubles)
 *   nxfx_residual_finish <- all-reduced buf: shared rows written back to r, nrm_out_d = [||r||^2,
 *                        ||b||^2], identical on every rank
 * Higher-order elements (nxfx_set_generic_system + nxfx_set_condensation) take the same calls; the
 * shared nodes then carry 2 x 2 blocks {P_b, lam_b} and the sections grow (nxfx_exchange_sizes):
 *   setup  [partial diagonal blocks D | coupling blocks U to the parent | L from the parent]
 *          12 max(n_shared, 1) doubles, 2 x 2 row-major per shared node (U, L of a link between two
 *          shared nodes come from rank 0, which holds that edge; the other ranks send zeros)
 *   apply  [partial nodal right-hand side {P, lam}]  2 max(n_shared, 1) doubles
 *   residual [lam rows of r | P rows of r | P rows of b | ||r||^2 | ||b||^2]  (continuous pressure;
 *          DG0: [lam rows of r | ||r||^2 | ||b||^2])
 * _setup_end / _apply_end compute the shared nodes from the all-reduced buffer alone, in an order
 * that is the same on every rank: the replicated nodal unknowns are bit-identical across ranks.
 * Shared right-hand-side rows ("stay additive"): with a continuous pressure the row nq + node of a
 * shared bifurcation is a PARTIAL sum on every rank, in b as assembled (each rank integrates f over
 * its own cells) as in A x.  The application reads these rows unweighted (the sum over the ranks is
 * the full row) and the multiplier rows weighted by lam_weight (replicated after _residual_finish;
 * zero in b).  nxfx_residual_finish therefore writes the multiplier rows back replicated and the
 * nodal pressure rows on the owner only (lam_weight 1, the others 0), and ||b||^2 takes the shared
 * P rows of b from the all-reduced buffer, so every shared row counts once in both norms.
 * The peer exchange (nxfx_comm_create) is flux degree 1 / pressure degree 0 only and returns
 * NXFX_ERR_UNSUPPORTED on such a ctx.                                                          */
int nxfx_set_shared(nxfx_ctx* ctx, int32_t n_shared, const int32_t* shared_lm_h,
                    const double* lam_weight_h);
/* Peer exchange over NVLink: with a communicator the library does the small SUM all-reduces itself.
 * The kernel that produces the partial sums (the top-chunk block of the fused factor+solve kernel,
 * the last block of the residual kernel) stores them into every rank's exchange buffer (cudaIpc-
 * mapped peer memory), raises a flag, waits for the other ranks and adds the contributions in rank
 * order.  nxfx_solve (ksp preonly, pc lu, one cell per edge) then runs the single-GPU launch
 * sequence -- assembly, ONE cooperative tree kernel, back-substitution, residual -- with no host
 * round trip and no NCCL call, and returns norms that are identical on every rank.  All ranks
 * must call nxfx_solve collectively.
 *   nxfx_comm_create   after nxfx_set_tree_schedule + nxfx_set_shared: allocates this rank's buffer,
 *                      handle_out_h receives NXFX_COMM_HANDLE_BYTES (a cudaIpcMemHandle_t)
 *   (the caller all-gathers the handles with whatever it has: torch.distributed, MPI, a file)
 *   nxfx_comm_connect  handles_all_h = nranks handles in rank order; maps the peers' buffers     */
#define NXFX_COMM_HANDLE_BYTES 64
int nxfx_comm_create(nxfx_ctx* ctx, int32_t rank, int32_t nranks, void* handle_out_h,
                     int32_t* slot_doubles);
int nxfx_comm_connect(nxfx_ctx* ctx, const void* handles_all_h);
/* Ranks that are contexts of ONE process (one host thread each, on one GPU or on several): after
 * nxfx_comm_create on every context, each rank calls nxfx_comm_connect_local with ctxs_h[r] = rank r's
 * context.  Rank r's buffer is used through its device pointer (no IPC handle).  Every context must
 * run on its own stream created with cudaStreamNonBlocking (nxfx_set_stream).
 *   different devices: peer access is enabled (NXFX_ERR_COMM if the devices cannot reach each other)
 *   same device: the cooperative tree grids of all ranks on it must be resident together (sum of
 *     their blocks <= blocks per SM x SMs), else NXFX_ERR_UNSUPPORTED before anything is launched;
 *     the back-substitution is then not launched as a programmatic dependent of the tree kernel
 * NXFX_ERR_INVALID if nranks, the rank order or the slot size disagree between the contexts.
 * Every rank gets the same answer: each checks all the devices of the group.                    */
int nxfx_comm_connect_local(nxfx_ctx* ctx, nxfx_ctx* const* ctxs_h, int32_t nranks);
int nxfx_comm_destroy(nxfx_ctx* ctx);
/* dst_d[i] = sum over r of src_h[r][i], i < n, added in rank order 0, 1, ... (bit-identical on every
 * rank): the in-process replacement of the SUM all-reduce between the begin/end halves below.  A
 * kernel on the ctx's stream; src_h = nranks device pointers readable from the ctx's device (peer
 * access to another device is enabled on first use).  The caller orders the producers of src before
 * this call and its consumers after it (events).                                                   */
int nxfx_group_sum(nxfx_ctx* ctx, const double* const* src_h, int32_t nranks, double* dst_d, int64_t n);
/* doubles of the exchanged sections of the host-driven path, for either element family:
 * setup (nxfx_pc_setup_begin), apply (nxfx_pc_apply_begin; _setup_apply_* take setup + apply, the
 * application's part at offset setup) and residual (nxfx_residual_partial).  P1/DG0: 2 nt, nt and
 * n_shared + 2 with nt = max(n_shared, 1).                                                          */
int nxfx_exchange_sizes(nxfx_ctx* ctx, int32_t* setup, int32_t* apply, int32_t* residual);
int nxfx_pc_setup_begin(nxfx_ctx* ctx, double* buf_d);
int nxfx_pc_setup_end(nxfx_ctx* ctx, double* buf_d);
int nxfx_pc_apply_begin(nxfx_ctx* ctx, const double* r_d, double* buf_d);
int nxfx_pc_apply_end(nxfx_ctx* ctx, const double* r_d, double* z_d, double* buf_d, int add);
int nxfx_pc_setup_apply_begin(nxfx_ctx* ctx, const double* r_d, double* buf_d);
int nxfx_pc_setup_apply_end(nxfx_ctx* ctx, const double* r_d, double* z_d, double* buf_d);
int nxfx_residual_partial(nxfx_ctx* ctx, const double* b_d, const double* x_d, double* r_d,
                          double* buf_d);
int nxfx_residual_finish(nxfx_ctx* ctx, const double* buf_d, double* r_d, double* nrm_out_d);

/* ---- post-processing ----------------------------------------------------------------------- *
 * Replaces Function.interpolate into the DG space in extract_global_flux: post_processing.py:36-51.
 * out_d [2*n_cells]: DG1 dofs (cell-wise [q(first vertex), q(second vertex)]).                       */
int nxfx_global_flux(nxfx_ctx* ctx, const double* x_d, double* out_d);

/* ---- gather of device-resident inputs and outputs ------------------------------------------ *
 *   dst_d[r*N + j] = src_d[row(r)*S + (S == N ? j : 0)],  r < n_rows, j < N,
 *   row(r) = map_d[r] (int32 device table) or r when map_d is NULL;  S in {1, N}.
 * One kernel on the ctx's stream, asynchronous.  Its uses:
 *   - a coefficient given as a CUDA tensor (HydraulicNetworkAssembler.compute_forms): per graph edge
 *     (S = 1) or per cell (S = N) -> per cell, N = cells_per_edge, n_rows = local edges; on a partitioned
 *     network map_d = the rank's global edge ids restricts a whole-network array to the local edges
 *     (the device counterpart of np.repeat and arr[global_edges] of the NumPy path);
 *   - the higher-order global flux of device Functions (post_processing.extract_global_flux):
 *     N = S = 1, map_d = the flux dof of every DG entry.
 * The caller orders the producer of src_d before the call (the ctx's stream or an event).            */
int nxfx_gather(nxfx_ctx* ctx, const double* src_d, const int32_t* map_d, int32_t S, int64_t n_rows,
                int32_t N, double* dst_d);

#ifdef __cplusplus
}
#endif
#endif /* NXFX_B200_H */
