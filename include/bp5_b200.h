/* bp5_b200.h -- C ABI of the B200-native BP5 / step-64 hot path.
 *
 * This is the drop-in boundary: a plain C interface (opaque handles, plain
 * pointers and sizes, int status codes, no C++/torch types) that a host
 * program written against the reference's deal.II-style classes binds to.
 * The header-only C++ facade in include/dealii_b200/ re-creates those classes
 * (PoissonOperator, MatrixFree, distributed::Vector, SolverCGFullMerge,
 * SolverControl ...) on top of it; INTEGRATION.md shows the binding.
 *
 * Every entry point names the reference interface it replaces (file:line in
 * peterrum/deal-and-ceed-on-gpu).  [UPSTREAM] marks deal.II members that the
 * reference calls but does not vendor.
 *
 * Conventions
 *   - every function returns BP5_OK (0) or an error code; bp5_last_error()
 *     gives the message for the calling thread.  No exception crosses the ABI.
 *   - the caller owns handles and frees them with the matching *_destroy.
 *   - all device work is enqueued on the context's stream; functions that
 *     return a value to the host synchronise that stream, the others do not.
 *   - vectors are [owned | ghost] contiguous in device memory
 *     (LinearAlgebra::distributed::Vector semantics, SURVEY.md section 5).
 *   - there is NO CPU fallback: without a CUDA device every compute entry
 *     point fails with BP5_ERR_CUDA.
 */
#ifndef BP5_B200_H
#define BP5_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bp5_context_s *bp5_context_t;
typedef struct bp5_operator_s *bp5_operator_t;
typedef struct bp5_vector_s *bp5_vector_t;

enum bp5_status {
  BP5_OK = 0,
  BP5_ERR_INVALID = 1,        /* bad argument / handle */
  BP5_ERR_CUDA = 2,           /* CUDA runtime error (message in bp5_last_error) */
  BP5_ERR_NO_CONVERGENCE = 3, /* SolverControl::NoConvergence, bp5/solver.h:540 */
  BP5_ERR_DIVIDE_BY_ZERO = 4, /* ExcDivideByZero, bp5/solver.h:501 */
  BP5_ERR_UNSUPPORTED = 5
};

enum { BP5_QUAD_GAUSS = 0, BP5_QUAD_GLL = 1 };     /* bp5/step-64.cu:243-247 (COLLOCATION) */
enum { BP5_OP_POISSON = 0, BP5_OP_HELMHOLTZ = 1 }; /* bp5/step-64.cu:147 ; step-64/step-64.cu:201 */
enum { BP5_GEOM_STORED = 0,      /* merged coefficient precomputed and streamed (evaluate_coefficients(JacobianFunctor), bp5/step-64.cu:256-258) */
       BP5_GEOM_ON_THE_FLY = 1 }; /* only nodal coordinates stored (24 B/DoF), the cell kernel rebuilds G (and a(x) JxW): both quadratures,    */
                                  /* both operators, affine and deformed meshes; not with refined meshes or the coloured cell order            */
enum { BP5_CELL_ORDER_DEFAULT = 0,  /* one pass, skeleton DoFs accumulated with atomics (use_coloring = false, bp5/step-64.cu:243) */
       BP5_CELL_ORDER_COLORED = 1 }; /* eight parity colours, one pass each, plain adds: bitwise reproducible (use_coloring = true) */
enum { BP5_CONTROL_ITERATION_NUMBER = 0, /* IterationNumberControl, bp5/step-64.cu:443 */
       BP5_CONTROL_SOLVER = 1 };         /* SolverControl, step-64/step-64.cu:513 */
enum { BP5_CG_STANDARD = 0,              /* dealii::SolverCG ("pcg-standard"), bp5/step-64.cu:446 */
       BP5_CG_MERGED = 1 };              /* SolverCGFullMerge ("pcg-merged"), bp5/solver.h:343 */

/* What the reference builds from GridGenerator::subdivided_hyper_rectangle +
 * refine_global + DoFHandler/FE_Q + MappingQGeneric + QGauss + zero Dirichlet
 * constraints (bp5/step-64.cu:228-259, 341-368, 656-663): a structured hex
 * mesh, optionally smoothly deformed, optionally one block of a Cartesian
 * partition (one block per GPU, replacing the p4est partition). */
typedef struct bp5_problem {
  int32_t degree;          /* fe_degree p, 1..8 */
  int32_t quadrature;      /* BP5_QUAD_* with p+1 points per direction */
  int32_t operator_kind;   /* BP5_OP_* */
  int32_t geometry_mode;   /* BP5_GEOM_* */
  int32_t cells[3];        /* global number of cells per direction */
  double lower[3];         /* domain corner */
  double upper[3];
  int32_t deformation;     /* 0 none; 1: x -> x + eps*L*prod_d sin(pi (x_d-lo_d)/L_d) */
  double deformation_eps;
  int32_t part_grid[3];    /* process grid (1,1,1 for one GPU) */
  int32_t part_coord[3];   /* this block's coordinates in the grid */
  int32_t cell_order;      /* BP5_CELL_ORDER_* (single block, stored geometry) */
  int32_t refine_lo[3];    /* locally refined mesh: the coarse cells with indices in [refine_lo, refine_hi) are replaced */
  int32_t refine_hi[3];    /* by their eight children (hanging nodes on the box's faces); all zero: conforming mesh.    */
                           /* vmult, cell_loop, assemble_rhs, l2_norm, the diagonal, the CG solves and                   */
                           /* bp5_operator_matrix_free_data (user functors) work on such an operator; the coefficient   */
                           /* export returns BP5_ERR_UNSUPPORTED.  Single block, stored geometry, default cell order.                  */
  int32_t reserved[1];     /* must be zero */
} bp5_problem_t;

/* ---- context ---------------------------------------------------------- */
/* replaces print_hardware_specs()/cudaSetDevice, bp5/step-64.cu:683-709 */
int bp5_context_create(int device, bp5_context_t *ctx);
int bp5_context_destroy(bp5_context_t ctx);
int bp5_context_synchronize(bp5_context_t ctx);
/* raw cudaStream_t of the context (for callers that interleave their own work) */
void *bp5_context_stream(bp5_context_t ctx);
const char *bp5_last_error(void);
const char *bp5_version(void);

/* ---- operator: PoissonOperator / HelmholtzOperator --------------------- */
/* ctor: PoissonOperator(dof_handler, constraints) bp5/step-64.cu:228-259
 * (MatrixFree::reinit :248, evaluate_coefficients(JacobianFunctor) :256-258);
 * HelmholtzOperator ctor step-64/step-64.cu:276-302. */
int bp5_operator_create(bp5_context_t ctx, const bp5_problem_t *problem, bp5_operator_t *op);
int bp5_operator_destroy(bp5_operator_t op);
/* sizes of a vector this operator works on: locally owned, ghost, global */
int bp5_operator_sizes(bp5_operator_t op, int64_t *n_owned, int64_t *n_ghost, int64_t *n_global,
                       int64_t *n_local_cells);
/* initialize_dof_vector, bp5/step-64.cu:210-215 */
int bp5_operator_initialize_dof_vector(bp5_operator_t op, bp5_vector_t *vec);
/* public member do_zero_out, bp5/step-64.cu:223 */
int bp5_operator_set_zero_out(bp5_operator_t op, int do_zero_out);
/* vmult(dst, src), bp5/step-64.cu:263-276: optional dst=0, cell loop
 * (ghost update, kernel, compress), copy_constrained_values. */
int bp5_operator_vmult(bp5_operator_t op, bp5_vector_t dst, bp5_vector_t src);
/* the two halves of vmult separately [UPSTREAM MatrixFree::cell_loop /
 * copy_constrained_values], called at bp5/step-64.cu:274-275 */
int bp5_operator_cell_loop(bp5_operator_t op, bp5_vector_t dst, bp5_vector_t src);
int bp5_operator_copy_constrained_values(bp5_operator_t op, bp5_vector_t dst, bp5_vector_t src);
/* raw device pointers, single block only (no ghosts): dst[n], src[n] */
int bp5_operator_vmult_ptr(bp5_operator_t op, double *dst_dev, const double *src_dev, int zero_dst);
/* assemble_rhs, bp5/step-64.cu:372-418: b_i = int phi_i, QGauss(p+1),
 * constrained rows zero; written to the owned range of b. */
int bp5_operator_assemble_rhs(bp5_operator_t op, bp5_vector_t b);
/* the merged coefficient in the REFERENCE layout coef[plane][cell][q],
 * planes xx,yy,zz,xy,xz,yz (bp5/step-64.cu:107-113), cells in this block's
 * lexicographic order, copied to host (for inspection/parity). 6*cells*n^3 doubles. */
int bp5_operator_export_coefficients(bp5_operator_t op, double *host_out);
/* coordinates (x,y,z) of the locally owned + ghost DoFs, host, 3 doubles each */
int bp5_operator_export_dof_coordinates(bp5_operator_t op, double *host_out);
/* global lexicographic index of each local (owned, then ghost) DoF, host */
int bp5_operator_export_global_indices(bp5_operator_t op, int64_t *host_out);
/* ||u||_L2 with QGauss(p+2), this block's contribution squared
 * (output_results, bp5/step-64.cu:604-615) */
int bp5_operator_l2_norm_sqr(bp5_operator_t op, bp5_vector_t u, double *out);
/* diagonal of the operator (Dirichlet rows: 1), or its reciprocal when invert != 0 -- the vector for a
 * Jacobi preconditioner in the DiagonalMatrix slot of the solvers (the reference passes ones,
 * bp5/step-64.cu:428-432).  Stored-metric operators.  On a partitioned mesh the ghost entries hold the
 * contributions for the neighbouring owners (compress(add) them, then invert). */
int bp5_operator_compute_diagonal(bp5_operator_t op, bp5_vector_t diag, int invert);
/* algorithmic bytes of one vmult over this block (SURVEY 8d: 16 + 48 r per DoF) */
int bp5_operator_algorithmic_bytes(bp5_operator_t op, double *bytes_per_vmult, double *bytes_per_cg_it);
/* live timing of the cell kernel: when enabled, every launch of the hot kernel
 * is bracketed by CUDA events on the context's stream; profile_result
 * synchronises, returns the number of launches and their summed device time
 * since the last call, and resets the counters. */
int bp5_operator_profile(bp5_operator_t op, int enable);
int bp5_operator_profile_result(bp5_operator_t op, int64_t *launches, double *total_ms);
/* name of the hand-written kernel variant chosen for this operator */
const char *bp5_operator_kernel_name(bp5_operator_t op);
/* number of kernels this library has launched on the context since creation */
int64_t bp5_context_launch_count(bp5_context_t ctx);

/* ---- vector: LinearAlgebra::distributed::Vector<double, CUDA> ---------- */
/* [UPSTREAM] used at bp5/step-64.cu:321-323,349,363-367 ; solver.h:369-382 */
int bp5_vector_create(bp5_context_t ctx, int64_t n_owned, int64_t n_ghost, bp5_vector_t *vec);
int bp5_vector_create_like(bp5_vector_t other, bp5_vector_t *vec); /* reinit(other) */
/* the operator whose initialize_dof_vector() produced this vector (directly or through
 * reinit(other)) -- the role the Partitioner plays in deal.II [UPSTREAM]; NULL for
 * vectors made by bp5_vector_create.  It must outlive the solves that use the vector. */
bp5_operator_t bp5_vector_owner(bp5_vector_t vec);
int bp5_vector_destroy(bp5_vector_t vec);
int bp5_vector_local_size(bp5_vector_t vec, int64_t *n_owned, int64_t *n_ghost);
double *bp5_vector_get_values(bp5_vector_t vec);                   /* get_values(): device pointer */
int bp5_vector_set(bp5_vector_t vec, double value);                /* operator=(double): owned and ghost */
int bp5_vector_import_host(bp5_vector_t vec, const double *host, int64_t n); /* import(rw, insert) */
int bp5_vector_export_host(bp5_vector_t vec, double *host, int64_t n);
int bp5_vector_copy(bp5_vector_t dst, bp5_vector_t src);
int bp5_vector_add(bp5_vector_t y, double a, bp5_vector_t x);      /* y.add(a, x) */
int bp5_vector_equ(bp5_vector_t y, double a, bp5_vector_t x);      /* y.equ(a, x) */
int bp5_vector_sadd(bp5_vector_t y, double s, double a, bp5_vector_t x); /* y = s*y + a*x */
int bp5_vector_scale(bp5_vector_t y, bp5_vector_t x);              /* y.scale(x): y[i] *= x[i] */
/* local (this block's owned range) parts of the reductions; the caller sums
 * over blocks (MPI_Allreduce in the reference, bp5/solver.h:493) */
int bp5_vector_dot_local(bp5_vector_t x, bp5_vector_t y, double *out);
int bp5_vector_norm_sqr_local(bp5_vector_t x, double *out);        /* l2_norm()^2 */
int bp5_vector_all_zero_local(bp5_vector_t x, int *out);           /* all_zero() */
int bp5_vector_zero_out_ghosts(bp5_vector_t vec);                  /* zero_out_ghosts() */

/* ---- solver ------------------------------------------------------------ */
/* SolverCGFullMerge::solve(A, x, b, preconditioner) bp5/solver.h:343-542 and
 * dealii::SolverCG::solve as used at bp5/step-64.cu:446-453.
 *   diag          DiagonalMatrix::get_vector() (solver.h:421) or NULL for the
 *                 identity (the reference passes a vector of ones, step-64.cu:432)
 *   tol           absolute tolerance on the residual l2 norm
 *   control       BP5_CONTROL_*; max_its its step limit
 *   last_step     SolverControl::last_step(); last_value its last_value()
 *   history       optional host array, history[it] = residual after it iterations
 * returns BP5_OK, BP5_ERR_NO_CONVERGENCE (x holds the last iterate) or an error.
 * Single block only; multi-block solves go through bp5_cg_* stepwise API below
 * driven by the host that owns the communicator. */
int bp5_cg_solve(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diag, int variant,
                 int control, double tol, int max_its, int *last_step, double *last_value,
                 double *history, int history_len);
/* same, with HOST buffers: copies b (and x0) to the device, solves, copies x
 * back -- the end-to-end entry point a host-side caller uses.
 *   x0_is_zero != 0: the initial guess is zero, as in the reference's drivers (solution = 0 before every
 *   solve, bp5/step-64.cu:449,491); x_host is then output only and is not uploaded. */
int bp5_cg_solve_host(bp5_operator_t op, double *x_host, const double *b_host, int64_t n, int x0_is_zero, int variant,
                      int control, double tol, int max_its, int *last_step, double *last_value);

/* ---- user-written cell functors (generic MatrixFree path) ------------------- */
/* What CUDAWrappers::MatrixFree<dim,double>::Data hands to a device functor
 * (bp5/step-64.cu:69-75,128-138; bp5/fe_evaluation_gl.h:107-124), in deal.II's layout:
 *   inv_jacobian[(d*3+e)*n_cells*padding_length + cell*padding_length + q] = d xi_d / d x_e
 *   JxW[cell*padding_length + q],  local_to_global[cell*padding_length + i],
 *   q_points[(cell*padding_length + q)*3 + c],  constraint_mask[cell] (0 on conforming meshes; see below),
 * plus the 1D shape tables [q*n + i] that MatrixFree::reinit puts into constant memory
 * [UPSTREAM]: values, gradients, and gradients of the basis through the quadrature points.
 * Device arrays stay owned by the operator.  Single block (no ghosts).
 * include/dealii_b200/cuda_matrix_free.cuh builds MatrixFree / FEEvaluationGL on this. */
typedef struct bp5_matrix_free_data {
  double *q_points;
  unsigned int *local_to_global;
  double *inv_jacobian;
  double *JxW;
  unsigned int *constraint_mask;
  unsigned int n_cells;
  unsigned int padding_length;
  int n_q_points_1d;
  int collocation;                 /* 1: Gauss-Lobatto quadrature on the nodes, shape_values == identity */
  double shape_values[81];
  double shape_gradients[81];
  double co_shape_gradients[81];
  /* locally refined meshes: [s][a*n + b] = value of the parent's 1D basis function b at node a of child s (s = 0, 1).
   * constraint_mask[cell]: bit d (0..2) = the cell's face normal to d that lies on its parent's boundary is
   * constrained (its nodes hold the unrefined neighbour's face DoFs and are interpolated by the evaluator);
   * bit 3+d = the cell's position s_d in its parent (low face if 0, high face if 1).  0 on conforming cells. */
  double hanging_interpolation[2][81];
} bp5_matrix_free_data_t;
int bp5_operator_matrix_free_data(bp5_operator_t op, bp5_matrix_free_data_t *out);
/* The same arrays for ONE of the eight parity colours of the cells (colour = px + 2 py + 4 pz, cells with
 * cx % 2 == px, ... in x-fastest order): cells of a colour share no DoF, so a cell loop over one colour may add
 * into dst with plain stores -- MatrixFree::AdditionalData::use_coloring / get_data(color) [UPSTREAM],
 * bp5/fe_evaluation_gl.h:176-177.  n_cells is that colour's cell count (0: nothing allocated). */
int bp5_operator_matrix_free_data_colored(bp5_operator_t op, int color, bp5_matrix_free_data_t *out);

/* ---- partitioned meshes: halo exchange and stepwise CG -------------------- */
/* Message shapes of update_ghost_values / compress(add) [UPSTREAM, inside cell_loop,
 * requested at bp5/step-64.cu:241].  Index m = 1..7 is a direction mask (bit d set: the
 * partner differs in dimension d); arrays have 8 entries, entry 0 unused.
 *   send_count/offset[m]: entries this block packs for its UPPER neighbour in direction m,
 *                         and where they sit in the packed send buffer;
 *   recv_count/offset[m]: ghost entries owned by the LOWER neighbour in direction m, and
 *                         where that (contiguous) group starts in the vector's ghost region. */
int bp5_operator_halo_info(bp5_operator_t op, int64_t *send_count, int64_t *send_offset, int64_t *recv_count,
                           int64_t *recv_offset);
/* update_ghost_values, sender side: sendbuf[offset[m] + t] = vec[owned dof t of group m].
 * The receiver needs no unpack: group m lands at vec + n_owned + recv_offset[m]. */
int bp5_operator_halo_pack(bp5_operator_t op, bp5_vector_t vec, double *sendbuf_dev);
/* compress(add), owner side: vec[owned dof t of group m] += recvbuf[offset[m] + t]
 * (the sender ships its ghost groups as they are, then calls bp5_vector_zero_out_ghosts). */
int bp5_operator_halo_unpack_add(bp5_operator_t op, bp5_vector_t vec, const double *recvbuf_dev);

/* SolverCGFullMerge::solve (bp5/solver.h:343-542) split at its communication points, for a
 * host that owns the communicator: per iteration it >= 1
 *   bp5_cg_step_update(op, it)          1) update region, solver.h:413-448
 *   [update_ghost_values(d)]            d, h, g from bp5_cg_step_vectors
 *   bp5_cg_step_apply_local(op)         2) h += local cells' part of A d, solver.h:475
 *   [compress(add)(h)]
 *   bp5_cg_step_constrained(op)            Dirichlet copy, bp5/step-64.cu:275
 *   bp5_cg_step_local_dots(op, s)       3) seven local sums, solver.h:478-485, left on the device
 *   [allreduce(s, 7 doubles, sum)]      4) MPI_Allreduce, solver.h:493
 *   bp5_cg_step_scalars(op, s)             alpha, beta, residual, stopping test, solver.h:497-533
 * Everything is enqueued on the context's stream; only bp5_cg_step_poll synchronises.  After the
 * stopping test fires every step becomes a no-op, so the host may poll every few iterations.
 * begin(): x must be zero (g = -b); res0 = global |b|_2 computed by the caller. */
int bp5_cg_step_begin(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diag, int control, double tol,
                      int max_its, double res0, int history_len);
int bp5_cg_step_vectors(bp5_operator_t op, bp5_vector_t *g, bp5_vector_t *d, bp5_vector_t *h);
int bp5_cg_step_update(bp5_operator_t op, int iteration);
int bp5_cg_step_apply_local(bp5_operator_t op);
int bp5_cg_step_constrained(bp5_operator_t op);
int bp5_cg_step_local_dots(bp5_operator_t op, double *sums7_dev);
int bp5_cg_step_scalars(bp5_operator_t op, const double *sums7_dev);
int bp5_cg_step_poll(bp5_operator_t op, int *state, int *last_step, double *last_value);
/* owed x update (solver.h:509-526); history (optional, host) receives history[1..] */
int bp5_cg_step_finish(bp5_operator_t op, double *history);

/* ---- peer-memory transport: blocks inside one NVLink / NVSwitch domain ------------------ */
/* One process per GPU.  Instead of CUDA-aware MPI (MPI_Isend/Irecv on device pointers inside
 * cell_loop [UPSTREAM], tests/cuda_aware_mpi.cc:29-46) and the host MPI_Allreduce of seven doubles
 * (bp5/solver.h:489-494), every exchange is done by kernels that store into the neighbour's memory
 * through CUDA IPC mappings and signal with flags; the cells that need no ghost data run while the
 * halo is in flight (overlap_communication_computation, bp5/step-64.cu:241).
 *   1. every rank: bp5_peer_export(op, rank, world, &info)      -> publish `info` to all ranks
 *      (any byte transport: MPI_Allgather, torch.distributed.all_gather_object, a file ...)
 *   2. every rank: bp5_peer_connect(op, all_infos, upper_rank, lower_rank)
 *      upper_rank[m] / lower_rank[m], m = 1..7 direction mask: the rank that receives this block's
 *      send group m / that owns its ghost group m, or -1
 *   3. a barrier of the caller's (all ranks connected) before the first exchange, and one before destroy
 *   4. bp5_peer_cg_solve / bp5_peer_vmult: collective calls, same arguments on every rank. */
typedef struct bp5_peer_info {
  unsigned char buf_handle[64];   /* cudaIpcMemHandle_t: landing zone, mailboxes, flags */
  unsigned char dvec_handle[64];  /* cudaIpcMemHandle_t: the vector whose ghost segments receive update_ghost_values */
  int64_t n_owned, n_ghost, n_send;
  int64_t ghost_offset[8];        /* start of ghost group m relative to n_owned */
  int64_t send_offset[8];         /* start of send group m in the landing zone */
  int32_t rank, device;
} bp5_peer_info_t;
int bp5_peer_export(bp5_operator_t op, int rank, int world, bp5_peer_info_t *info);
int bp5_peer_connect(bp5_operator_t op, const bp5_peer_info_t *all_infos, const int32_t *upper_rank,
                     const int32_t *lower_rank);
/* dst = A src over the partition (owned range of dst; vmult, bp5/step-64.cu:263-276) */
int bp5_peer_vmult(bp5_operator_t op, bp5_vector_t dst, bp5_vector_t src);
/* SolverCGFullMerge::solve over the partition; x must be zero on entry (the reference's use,
 * bp5/step-64.cu:491); arguments and results as bp5_cg_solve, identical on every rank */
int bp5_peer_cg_solve(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diag, int control, double tol,
                      int max_its, int *last_step, double *last_value, double *history, int history_len);
/* in-place sum over all ranks of n <= 8 host values (l2_norm and friends, bp5/solver.h:382) */
int bp5_peer_allreduce(bp5_operator_t op, double *values, int n);
/* number of ranks this operator's peer transport is connected to (1: single block / not connected) */
int bp5_peer_world_size(bp5_operator_t op);
/* Ghost-value semantics of LinearAlgebra::distributed::Vector [UPSTREAM] for ANY vector of this operator's layout
 * (the reference relies on them inside cell_loop, bp5/step-64.cu:241,272-275, and on vectors made by
 * reinit(owned, relevant, comm), :349,363-366).  Collective: every rank calls, in the same order.
 *   update_ghost_values: ghost entries <- the owners' values;
 *   compress_add:        owners' entries += the ghost entries of the neighbours, ghost entries <- 0
 *                        (compress(VectorOperation::add) followed by zero_out_ghosts, as cell_loop leaves dst). */
int bp5_vector_update_ghost_values(bp5_operator_t op, bp5_vector_t vec);
int bp5_vector_compress_add(bp5_operator_t op, bp5_vector_t vec);
/* bp5_peer_cg_solve with HOST buffers of this block's owned range (n = n_owned): b in, x out (and x in unless
 * x0_is_zero) -- the reference imports the right-hand side from the host and exports the solution
 * (bp5/step-64.cu:415-417,553-555).  Collective. */
int bp5_peer_cg_solve_host(bp5_operator_t op, double *x_host, const double *b_host, int64_t n, int x0_is_zero,
                           int control, double tol, int max_its, int *last_step, double *last_value);

/* ---- geometric multigrid: Chebyshev-Jacobi V-cycle as a CG preconditioner ------------------ */
/* The setup deal.II users pair with a matrix-free operator (MGTransferMatrixFree + PreconditionChebyshev +
 * MGCoarseGridIterativeSolver inside PreconditionMG) for one block, conforming mesh, stored geometry, default cell
 * order: every other operator gets BP5_ERR_UNSUPPORTED from bp5_mg_create.
 *   levels      level n_levels-1 is the caller's operator (not owned; it must outlive the multigrid object); level
 *               l-1 is the same problem with every cells[d] halved, down to a mesh with an odd or unit cell count
 *               (or max_levels levels).
 *   transfer    prolongation P = nodal interpolation coarse -> fine (P_z (x) P_y (x) P_x on the DoF lattice),
 *               restriction R = P^T followed by zeroed Dirichlet rows; no atomics, bitwise repeatable.
 *   smoother    Chebyshev iteration of the given degree with D^-1 (inverse diagonal) on levels >= 1, eigenvalue
 *               range [1.2 lambda / smoothing_range, 1.2 lambda], lambda estimated at set-up by eig_iterations
 *               Jacobi-preconditioned CG (Lanczos) steps on D^-1 A from a fixed-seed start vector.
 *   coarse      level 0: standard CG with Jacobi to coarse_tol * |b| or coarse_max_its steps (running out of steps
 *               is not an error).
 * Zero in a field of bp5_mg_params_t selects the default; reserved fields must be zero. */
typedef struct bp5_mg_s *bp5_mg_t;
typedef struct bp5_mg_params {
  int32_t max_levels;       /* 0: as many as the mesh allows */
  int32_t smoothing_degree; /* PreconditionChebyshev::AdditionalData::degree, default 5 */
  double smoothing_range;   /* ::smoothing_range, default 15 */
  int32_t eig_iterations;   /* ::eig_cg_n_iterations, default 12 */
  int32_t coarse_max_its;   /* default 1000 */
  double coarse_tol;        /* relative, default 1e-6 */
  int32_t reserved[4];
} bp5_mg_params_t;
/* MGLevelObject + MGTransferMatrixFree::build + PreconditionChebyshev::initialize per level [UPSTREAM];
 * params may be NULL (all defaults) */
int bp5_mg_create(bp5_operator_t fine_op, const bp5_mg_params_t *params, bp5_mg_t *mg);
int bp5_mg_destroy(bp5_mg_t mg);
int bp5_mg_n_levels(bp5_mg_t mg, int *n_levels);
/* the operator of a level (non-owning; level n_levels-1 is the caller's) */
int bp5_mg_level_operator(bp5_mg_t mg, int level, bp5_operator_t *op);
/* PreconditionChebyshev's estimate of the largest eigenvalue of D^-1 A on a level >= 1 (before the factor 1.2);
 * set replaces it (the smoother then uses the new value) */
int bp5_mg_get_lambda_max(bp5_mg_t mg, int level, double *lambda);
int bp5_mg_set_lambda_max(bp5_mg_t mg, int level, double lambda);
/* MGTransferMatrixFree::prolongate: dst (level fine_level) = P src (level fine_level-1) */
int bp5_mg_prolongate(bp5_mg_t mg, int fine_level, bp5_vector_t dst, bp5_vector_t src);
/* MGTransferMatrixFree::restrict_and_add into a zeroed dst: dst (level fine_level-1) = R src, Dirichlet rows 0 */
int bp5_mg_restrict(bp5_mg_t mg, int fine_level, bp5_vector_t dst, bp5_vector_t src);
/* PreconditionChebyshev::step on a level >= 1: x <- Chebyshev smoothing of A x = b from the x given (an all-zero x
 * takes the path without the initial operator application) */
int bp5_mg_smooth(bp5_mg_t mg, int level, bp5_vector_t x, bp5_vector_t b);
/* PreconditionMG::vmult: dst = V(src), one V-cycle from a zero initial guess on the finest level */
int bp5_mg_vcycle(bp5_mg_t mg, bp5_vector_t dst, bp5_vector_t src);
/* dealii::SolverCG::solve(A, x, b, PreconditionMG) on the finest level; arguments, status codes and history as
 * bp5_cg_solve (x on entry is the initial guess).  Scalars live on the host: one V-cycle per iteration. */
int bp5_mg_cg_solve(bp5_mg_t mg, bp5_vector_t x, bp5_vector_t b, int control, double tol, int max_its, int *last_step,
                    double *last_value, double *history, int history_len);
/* timing of the V-cycle's parts by CUDA events on the context's stream (off by default).  profile_result
 * synchronises, writes ms[4 * level + k] for k = 0 operator applications, 1 transfers between the level and the next
 * coarser one (restriction, zeroed Dirichlet rows, prolongation), 2 Chebyshev and residual vector kernels, 3 coarse
 * solve (level 0 only),
 * returns the number of V-cycles since the last call and resets the counters. */
int bp5_mg_profile(bp5_mg_t mg, int enable);
int bp5_mg_profile_result(bp5_mg_t mg, double *ms, int64_t *n_vcycles);

#ifdef __cplusplus
}
#endif
#endif /* BP5_B200_H */
