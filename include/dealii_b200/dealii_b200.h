// dealii_b200.h -- header-only C++ facade over the C ABI (include/bp5_b200.h).
//
// Re-creates, for the BP5 / step-64 hot path only, the deal.II-style host
// interface the reference is written against, so that driver and solver code
// shaped like bp5/step-64.cu and bp5/solver.h compiles against this library:
//
//   BP5::PoissonOperator<dim, fe_degree>            bp5/step-64.cu:198-276
//   Step64::HelmholtzOperator<dim, fe_degree>       step-64/step-64.cu:232-322
//   LinearAlgebra::distributed::Vector<double, MemorySpace::CUDA>   [UPSTREAM]
//        (bp5/step-64.cu:321-323,349,363-367,417,432,445; solver.h:352-382,405,417,511)
//   SolverControl / IterationNumberControl           bp5/step-64.cu:443-445,460
//   SolverCG, SolverCGFullMerge                      bp5/step-64.cu:446-453; solver.h:15-31
//   DiagonalMatrix                                   bp5/step-64.cu:428-432
//   Triangulation / GridGenerator::subdivided_hyper_rectangle / DoFHandler / FE_Q /
//   AffineConstraints: only as far as the drivers use them to DESCRIBE the
//   structured mesh (bp5/step-64.cu:341-368,656-663); the mesh itself is
//   generated on the GPU by the library.
//
// Errors: every C status code is turned back into the C++ exception the
// reference throws (SolverControl::NoConvergence, ExcDivideByZero, ...).
// One host thread per GPU, one stream per context (the reference uses the
// default stream and one MPI rank per GPU, bp5/step-64.cu:704-707,720).
#pragma once

#include <array>
#include <chrono>
#include <cmath>
#include <iostream>
#include <memory>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "../bp5_b200.h"

namespace dealii {

namespace types { using global_dof_index = unsigned int; }
namespace VectorOperation { enum values { unknown, insert, add }; }
namespace MemorySpace { struct Host {}; struct CUDA {}; }

struct ExcMessage : std::runtime_error { using std::runtime_error::runtime_error; };
struct ExcDivideByZero : std::runtime_error { ExcDivideByZero() : std::runtime_error("ExcDivideByZero") {} };

// ------------------------------------------------------------------ SolverControl
class SolverControl {
 public:
  enum State { iterate = 0, success, failure };
  class NoConvergence : public std::runtime_error {
   public:
    NoConvergence(unsigned int step, double residual)
        : std::runtime_error("Iterative method reported convergence failure in step " + std::to_string(step) +
                             ". The residual in the last step was " + std::to_string(residual) + "."),
          last_step(step), last_residual(residual) {}
    const unsigned int last_step;
    const double last_residual;
  };
  SolverControl(unsigned int n = 100, double tol = 1e-10) : maxsteps(n), tol(tol) {}
  virtual ~SolverControl() = default;
  unsigned int last_step() const { return lstep; }
  double last_value() const { return lvalue; }
  double tolerance() const { return tol; }
  unsigned int max_steps() const { return maxsteps; }
  virtual int abi_kind() const { return BP5_CONTROL_SOLVER; }          // failure at max_steps
  void record(unsigned int step, double value) { lstep = step; lvalue = value; }

 protected:
  unsigned int maxsteps;
  double tol;
  unsigned int lstep = 0;
  double lvalue = 0.0;
};

// success at the tolerance OR at max_steps (bp5/step-64.cu:443-445)
class IterationNumberControl : public SolverControl {
 public:
  using SolverControl::SolverControl;
  int abi_kind() const override { return BP5_CONTROL_ITERATION_NUMBER; }
};

// ------------------------------------------------------------------ context
namespace b200 {
inline void check(int rc) {
  if (rc == BP5_OK) return;
  const std::string msg = bp5_last_error();
  if (rc == BP5_ERR_DIVIDE_BY_ZERO) throw ExcDivideByZero();
  throw ExcMessage("bp5_b200 error " + std::to_string(rc) + ": " + msg);
}
// one context per process: device = rank % n_devices (bp5/step-64.cu:704-707).  Call set_device() before the
// first library object is made (the reference calls cudaSetDevice at the top of main); default: device 0.
class Context {
 public:
  static void set_device(int device) { requested_device() = device; }
  static bp5_context_t get() {
    static Context c(requested_device());
    return c.h;
  }
  static void synchronize() { check(bp5_context_synchronize(get())); }   // cudaDeviceSynchronize in the driver

 private:
  static int &requested_device() { static int d = 0; return d; }
  explicit Context(int device) { check(bp5_context_create(device, &h)); }
  ~Context() { bp5_context_destroy(h); }
  bp5_context_t h = nullptr;
};

// What MPI_COMM_WORLD is to the reference (bp5/step-64.cu:349,363-366,720): one rank per GPU inside one NVLink
// domain.  Only the set-up travels through it (a few hundred bytes of CUDA IPC handles per rank and barriers):
// implement it over MPI_Allgather / MPI_Barrier in an MPI program, or over shared memory between forked
// processes (examples/bp5_step64_multi.cc).  The data plane -- halo exchange, sums of the CG scalars -- is the
// library's peer-memory transport (bp5_peer_*).
class Communicator {
 public:
  virtual ~Communicator() = default;
  virtual int rank() const = 0;
  virtual int size() const = 0;
  virtual void allgather(const void *send, void *recv_all, std::size_t bytes_per_rank) = 0;
  virtual void barrier() = 0;
};

// 1x1x1, 2x1x1, 2x2x1, 2x2x2 (SURVEY.md 8e); otherwise the most cubic factorisation, x >= y >= z
inline std::array<int, 3> process_grid(int world) {
  std::array<int, 3> best{world, 1, 1};
  int best_spread = world, best_px = world;
  for (int pz = 1; pz <= world; ++pz) {
    if (world % pz) continue;
    for (int py = pz; py <= world / pz; ++py) {
      if ((world / pz) % py) continue;
      const int px = world / (pz * py);
      if (px < py) continue;
      if (px - pz < best_spread || (px - pz == best_spread && px < best_px)) {
        best_spread = px - pz; best_px = px; best = {px, py, pz};
      }
    }
  }
  return best;
}
}  // namespace b200

// ------------------------------------------------------------------ mesh description
#ifdef __CUDACC__
#define DEAL_II_B200_HOST_DEVICE __host__ __device__
#else
#define DEAL_II_B200_HOST_DEVICE
#endif
template <int dim, typename Number = double> struct Point {
  Number v[dim] = {};
  DEAL_II_B200_HOST_DEVICE Number &operator[](unsigned d) { return v[d]; }
  DEAL_II_B200_HOST_DEVICE Number operator[](unsigned d) const { return v[d]; }
};

// what the drivers do to a parallel::distributed::Triangulation (bp5/step-64.cu:656-663)
template <int dim> class Triangulation {
 public:
  virtual ~Triangulation() = default;     // the operators dynamic_cast it (bp5/step-64.cu:250)
  void clear() { subdivisions.assign(dim, 1); refinements = 0; for (int d = 0; d < 3; ++d) refine_lo[d] = refine_hi[d] = 0; }
  // one block per GPU; this facade drives one block
  unsigned int n_locally_owned_active_cells() const { return (unsigned int)n_global_active_cells(); }
  void refine_global(unsigned int n) { refinements += n; }
  unsigned long long n_global_active_cells() const {
    unsigned long long n = 1, box = 1;
    for (int d = 0; d < dim; ++d) { n *= cells(d); box *= (unsigned long long)(refine_hi[d] - refine_lo[d]); }
    return n + 7 * box;
  }
  // Local refinement, one level: what flagging every cell with (x-fastest lattice) index in [lo, hi) and calling
  // execute_coarsening_and_refinement() does in deal.II -- those cells are replaced by their eight children, and the
  // children's faces on the box's surface carry hanging nodes, which both paths resolve: CUDAWrappers::MatrixFree +
  // FEEvaluationGL (constraint_mask / resolve_hanging_nodes, bp5/fe_evaluation_gl.h:88,150,167) and the tuned
  // BP5::PoissonOperator / Step64::HelmholtzOperator.  One block (no communicator).  Call after refine_global.
  void refine_cells_in_box(const std::array<unsigned int, 3> &lo, const std::array<unsigned int, 3> &hi) {
    for (int d = 0; d < 3; ++d) {
      if (!(lo[d] < hi[d] && hi[d] <= cells(d))) throw ExcMessage("refine_cells_in_box: need lo < hi <= cells");
      refine_lo[d] = (int)lo[d]; refine_hi[d] = (int)hi[d];
    }
  }
  bool locally_refined() const { return refine_hi[0] > refine_lo[0]; }
  int refine_lo[3] = {0, 0, 0}, refine_hi[3] = {0, 0, 0};
  unsigned int cells(int d) const { return subdivisions[d] << refinements; }
  std::vector<unsigned int> subdivisions = std::vector<unsigned int>(dim, 1);
  Point<dim> p1, p2;
  unsigned int refinements = 0;
  // smooth deformation of the mesh (BASELINE config 5; not in the reference)
  int deformation = 0;
  double deformation_eps = 0.0;
  // parallel::distributed::Triangulation<dim>(MPI_COMM_WORLD) (bp5/step-64.cu:310): the mesh is split into a
  // Cartesian grid of blocks, one per rank of the communicator (nullptr: one block)
  b200::Communicator *communicator = nullptr;
  explicit Triangulation(b200::Communicator *comm = nullptr) : communicator(comm) {}
};
namespace parallel {
template <int dim> using Triangulation = dealii::Triangulation<dim>;
namespace distributed { template <int dim> using Triangulation = dealii::Triangulation<dim>; }
}  // namespace parallel

namespace GridGenerator {
template <int dim>
void subdivided_hyper_rectangle(Triangulation<dim> &tria, const std::vector<unsigned int> &subdivisions,
                                const Point<dim> &p1, const Point<dim> &p2) {
  tria.subdivisions = subdivisions; tria.p1 = p1; tria.p2 = p2; tria.refinements = 0;
}
template <int dim> void hyper_cube(Triangulation<dim> &tria, double a = 0., double b = 1.) {
  Point<dim> p1, p2;
  for (int d = 0; d < dim; ++d) { p1[d] = a; p2[d] = b; }
  subdivided_hyper_rectangle(tria, std::vector<unsigned int>(dim, 1), p1, p2);
}
}  // namespace GridGenerator

template <int dim> struct FE_Q {
  explicit FE_Q(unsigned int degree) : degree(degree), dofs_per_cell(1) {
    for (int d = 0; d < dim; ++d) dofs_per_cell *= degree + 1;
  }
  unsigned int degree, dofs_per_cell;
};

template <int dim> class DoFHandler {
 public:
  explicit DoFHandler(const Triangulation<dim> &tria) : tria(&tria) {}
  void distribute_dofs(const FE_Q<dim> &fe) { degree = fe.degree; }
  unsigned long long n_dofs() const {
    unsigned long long n = 1;
    for (int d = 0; d < dim; ++d) n *= (unsigned long long)tria->cells(d) * degree + 1;
    if (tria->locally_refined()) {
      // minus the coarse nodes that only refined cells touch, plus the children's nodes that are not hanging
      unsigned long long gone = 1, fine = 1;
      for (int d = 0; d < dim; ++d) {
        const unsigned long long lo = tria->refine_lo[d], hi = tria->refine_hi[d];
        const unsigned long long faces = (lo > 0 ? 1 : 0) + (hi < tria->cells(d) ? 1 : 0);
        gone *= (hi - lo) * degree + 1 - faces;
        fine *= 2 * (hi - lo) * degree + 1 - faces;
      }
      n = n - gone + fine;
    }
    return n;
  }
  const Triangulation<dim> &get_triangulation() const { return *tria; }
  unsigned int degree = 1;

 private:
  const Triangulation<dim> *tria;
};

// quadrature / mapping descriptions as the operator constructors name them (bp5/step-64.cu:234-247)
template <int dim> struct Quadrature {
  Quadrature(unsigned int n, int kind) : n_points_1d(n), abi_kind(kind) {}
  unsigned int n_points_1d;
  int abi_kind;
};
template <int dim> struct QGauss : Quadrature<dim> {
  explicit QGauss(unsigned int n) : Quadrature<dim>(n, BP5_QUAD_GAUSS) {}
};
template <int dim> struct QGaussLobatto : Quadrature<dim> {
  explicit QGaussLobatto(unsigned int n) : Quadrature<dim>(n, BP5_QUAD_GLL) {}
};
template <int dim> struct MappingQGeneric {
  explicit MappingQGeneric(unsigned int degree) : degree(degree) {}
  unsigned int degree;
};
enum UpdateFlags { update_default = 0, update_values = 1, update_gradients = 2, update_JxW_values = 4, update_quadrature_points = 8 };
inline UpdateFlags operator|(UpdateFlags a, UpdateFlags b) { return static_cast<UpdateFlags>(int(a) | int(b)); }

// zero Dirichlet values on the whole boundary (boundary id 0), bp5/step-64.cu:351-358
template <typename Number = double> struct AffineConstraints {
  void clear() {}
  void close() {}
};

// ------------------------------------------------------------------ vector
namespace LinearAlgebra { namespace distributed {
template <typename Number, typename MemorySpaceType = MemorySpace::CUDA> class Vector;

template <> class Vector<double, MemorySpace::CUDA> {
 public:
  using value_type = double;
  using size_type = types::global_dof_index;
  Vector() = default;
  Vector(const Vector &) = delete;
  Vector &operator=(const Vector &) = delete;
  ~Vector() { release(); }

  void reinit(long long n_owned, long long n_ghost = 0) {
    release();
    b200::check(bp5_vector_create(b200::Context::get(), n_owned, n_ghost, &h));
    constant = 0.0; is_constant = true;
  }
  void reinit(const Vector &other, bool = false) {          // solver.h:369-371, bp5/step-64.cu:367,431
    release();
    b200::check(bp5_vector_create_like(other.h, &h));
    constant = 0.0; is_constant = true;
  }
  void adopt(bp5_vector_t handle) { release(); h = handle; constant = 0.0; is_constant = true; }
  // non-owning alias of a vector that lives in the library (the solver's temporaries)
  void view(bp5_vector_t handle) { release(); h = handle; owning = false; is_constant = false; }
  Vector &operator=(double s) { b200::check(bp5_vector_set(h, s)); constant = s; is_constant = true; return *this; }
  // reductions are over all blocks of the partition (MPI_Allreduce in deal.II [UPSTREAM]): local part on this
  // GPU, then the peer transport's all-rank sum; identical result on every rank
  double l2_norm() const { double v; b200::check(bp5_vector_norm_sqr_local(h, &v)); return std::sqrt(global_sum(v)); }
  double operator*(const Vector &o) const { double v; b200::check(bp5_vector_dot_local(h, o.h, &v)); return global_sum(v); }
  bool all_zero() const { int z; b200::check(bp5_vector_all_zero_local(h, &z)); return global_sum(z ? 0.0 : 1.0) == 0.0; }
  // ghost-value semantics (collective over the partition; no-ops on a single block):
  // update_ghost_values / compress(VectorOperation::add) [UPSTREAM], requested inside cell_loop at
  // bp5/step-64.cu:241,272-275
  void update_ghost_values() const { if (partitioned()) b200::check(bp5_vector_update_ghost_values(bp5_vector_owner(h), h)); }
  void compress(VectorOperation::values operation = VectorOperation::add) {
    if (operation != VectorOperation::add) throw ExcMessage("compress: only VectorOperation::add has an exchange here");
    if (partitioned()) b200::check(bp5_vector_compress_add(bp5_vector_owner(h), h));
    is_constant = false;
  }
  bool partitioned() const { bp5_operator_t op = bp5_vector_owner(h); return op != nullptr && bp5_peer_world_size(op) > 1; }
  void add(double a, const Vector &v) { b200::check(bp5_vector_add(h, a, v.h)); is_constant = false; }
  void equ(double a, const Vector &v) { b200::check(bp5_vector_equ(h, a, v.h)); is_constant = false; }
  void sadd(double s, double a, const Vector &v) { b200::check(bp5_vector_sadd(h, s, a, v.h)); is_constant = false; }
  void scale(const Vector &v) { b200::check(bp5_vector_scale(h, v.h)); is_constant = false; }
  void zero_out_ghosts() { b200::check(bp5_vector_zero_out_ghosts(h)); }
  double *get_values() { is_constant = false; return bp5_vector_get_values(h); }
  const double *get_values() const { return bp5_vector_get_values(h); }
  size_type local_size() const { int64_t a = 0, g = 0; bp5_vector_local_size(h, &a, &g); return (size_type)a; }
  size_type size() const {                              // global size, like deal.II's Vector::size()
    bp5_operator_t op = bp5_vector_owner(h);
    if (!op) return local_size();
    int64_t n_global = 0;
    bp5_operator_sizes(op, nullptr, nullptr, &n_global, nullptr);
    return (size_type)n_global;
  }
  // import(ReadWriteVector, insert) / the reverse, bp5/step-64.cu:415-417,553-555
  void import_from_host(const std::vector<double> &v) {
    b200::check(bp5_vector_import_host(h, v.data(), (int64_t)v.size())); is_constant = false;
  }
  void copy_to_host(std::vector<double> &v) const {
    v.resize(local_size());
    b200::check(bp5_vector_export_host(h, v.data(), (int64_t)v.size()));
  }
  double global_sum(double v) const {
    if (!partitioned()) return v;
    b200::check(bp5_peer_allreduce(bp5_vector_owner(h), &v, 1));
    return v;
  }
  bp5_vector_t handle() const { return h; }
  void mark_modified() { is_constant = false; }
  bool is_constant_value(double s) const { return is_constant && constant == s; }

 private:
  void release() { if (owning) bp5_vector_destroy(h); h = nullptr; owning = true; }
  bp5_vector_t h = nullptr;
  bool owning = true;
  double constant = 0.0;     // set by operator=(double) until the next modification
  bool is_constant = false;
};
} }  // namespace LinearAlgebra::distributed

template <typename VectorType> class DiagonalMatrix {
 public:
  VectorType &get_vector() { return diagonal; }
  const VectorType &get_vector() const { return diagonal; }

 private:
  VectorType diagonal;
};

// ------------------------------------------------------------------ operators
namespace b200 {
template <int dim, int fe_degree, int operator_kind> class MatrixFreeOperator {
  static_assert(dim == 3, "the hot path is three-dimensional");
 public:
  using VectorType = LinearAlgebra::distributed::Vector<double, MemorySpace::CUDA>;
  // use_coloring: MatrixFree::AdditionalData::use_coloring (bp5/step-64.cu:243 passes false): eight colour passes
  // with plain adds in place of the atomics, bitwise reproducible results (one block, stored geometry)
  MatrixFreeOperator(const DoFHandler<dim> &dof_handler, const AffineConstraints<double> &, int quadrature,
                     bool use_coloring = false)
      : do_zero_out(true) {
    const Triangulation<dim> &t = dof_handler.get_triangulation();
    bp5_problem_t pr{};
    pr.degree = fe_degree; pr.quadrature = quadrature; pr.operator_kind = operator_kind;
    for (int d = 0; d < 3; ++d) { pr.refine_lo[d] = t.refine_lo[d]; pr.refine_hi[d] = t.refine_hi[d]; }
    pr.geometry_mode = BP5_GEOM_STORED;
    pr.cell_order = use_coloring ? BP5_CELL_ORDER_COLORED : BP5_CELL_ORDER_DEFAULT;
    comm = t.communicator;
    const int world = comm ? comm->size() : 1, rank = comm ? comm->rank() : 0;
    const std::array<int, 3> grid = process_grid(world);
    const int coord[3] = {rank % grid[0], (rank / grid[0]) % grid[1], rank / (grid[0] * grid[1])};
    for (int d = 0; d < 3; ++d) {
      pr.cells[d] = (int32_t)t.cells(d); pr.lower[d] = t.p1[d]; pr.upper[d] = t.p2[d];
      pr.part_grid[d] = grid[d]; pr.part_coord[d] = coord[d];
    }
    pr.deformation = t.deformation; pr.deformation_eps = t.deformation_eps;
    check(bp5_operator_create(Context::get(), &pr, &h));
    if (world > 1) connect_peers(grid.data(), coord, world, rank);
  }
  MatrixFreeOperator(const MatrixFreeOperator &) = delete;
  ~MatrixFreeOperator() {
    if (comm && comm->size() > 1) {        // nobody unmaps while a neighbour may still store into this block
      bp5_context_synchronize(Context::get());
      comm->barrier();
    }
    bp5_operator_destroy(h);
  }

  void vmult(VectorType &dst, const VectorType &src) const {       // bp5/step-64.cu:263-276
    if (partitioned()) {
      // update_ghost_values(src) / cell loop with interior-boundary overlap / compress(add)(dst) / Dirichlet
      // copy, all by the peer transport's kernels.  (dst is overwritten: with do_zero_out == false the
      // reference accumulates into whatever dst held, which is only ever zero or garbage, SURVEY 3.4.)
      check(bp5_peer_vmult(h, dst.handle(), src.handle()));
    } else {
      check(bp5_operator_set_zero_out(h, do_zero_out));
      check(bp5_operator_vmult(h, dst.handle(), src.handle()));
    }
    dst.mark_modified();
  }
  bool partitioned() const { return comm != nullptr && comm->size() > 1; }
  void initialize_dof_vector(VectorType &vec) const {             // bp5/step-64.cu:210-215
    bp5_vector_t v = nullptr;
    check(bp5_operator_initialize_dof_vector(h, &v));
    vec.adopt(v);
  }
  // assemble_rhs of the drivers (bp5/step-64.cu:372-418), done on the device
  void assemble_rhs(VectorType &b) const { check(bp5_operator_assemble_rhs(h, b.handle())); b.mark_modified(); }
  // MatrixFreeOperators-style compute_diagonal(): fills a DiagonalMatrix's vector with the inverse diagonal
  void compute_inverse_diagonal(VectorType &diag) const {
    check(bp5_operator_compute_diagonal(h, diag.handle(), 1));
    diag.mark_modified();
  }
  // VectorTools::integrate_difference(..., L2_norm) + compute_global_error of output_results
  // (bp5/step-64.cu:604-615), on the device
  double l2_norm(const VectorType &u) const {
    double v = 0.0;
    u.update_ghost_values();               // the cells of a block read its ghost DoFs
    check(bp5_operator_l2_norm_sqr(h, u.handle(), &v));
    return std::sqrt(u.global_sum(v));
  }
  bp5_operator_t handle() const { return h; }

 private:
  // bp5_peer_export -> allgather of the handles -> bp5_peer_connect -> barrier (include/bp5_b200.h)
  void connect_peers(const int *grid, const int *coord, int world, int rank) {
    bp5_peer_info_t mine;
    check(bp5_peer_export(h, rank, world, &mine));
    std::vector<bp5_peer_info_t> all((std::size_t)world);
    comm->allgather(&mine, all.data(), sizeof(bp5_peer_info_t));
    int32_t upper[8], lower[8];
    for (int m = 0; m < 8; ++m) {
      upper[m] = lower[m] = -1;
      if (m == 0) continue;
      int cu[3], cl[3];
      bool has_u = true, has_l = true;
      for (int d = 0; d < 3; ++d) {
        const int bit = (m >> d) & 1;
        cu[d] = coord[d] + bit; cl[d] = coord[d] - bit;
        if (cu[d] >= grid[d]) has_u = false;
        if (cl[d] < 0) has_l = false;
      }
      if (has_u) upper[m] = cu[0] + grid[0] * (cu[1] + grid[1] * cu[2]);
      if (has_l) lower[m] = cl[0] + grid[0] * (cl[1] + grid[1] * cl[2]);
    }
    check(bp5_peer_connect(h, all.data(), upper, lower));
    check(bp5_context_synchronize(Context::get()));
    comm->barrier();
  }
  bp5_operator_t h = nullptr;
  Communicator *comm = nullptr;

 public:
  bool do_zero_out;                                               // bp5/step-64.cu:223
};

// PreconditionMG<dim, VectorType, MGTransferMatrixFree> with PreconditionChebyshev smoothers (Jacobi inside) and an
// MGCoarseGridIterativeSolver (CG) [UPSTREAM], all on the library's levels of the operator's mesh: one block,
// conforming mesh, stored geometry, default cell order.  The operator must outlive the preconditioner.
template <int dim, int fe_degree, int operator_kind> class MultigridPreconditioner {
 public:
  using VectorType = LinearAlgebra::distributed::Vector<double, MemorySpace::CUDA>;
  struct AdditionalData {                 // field names of PreconditionChebyshev::AdditionalData where they exist
    unsigned int degree = 5;
    double smoothing_range = 15.;
    unsigned int eig_cg_n_iterations = 12;
    unsigned int max_levels = 0;          // 0: coarsen while every cell count is even
    double coarse_tolerance = 1e-6;       // relative, MGCoarseGridIterativeSolver's SolverControl
    unsigned int coarse_max_iterations = 1000;
  };
  explicit MultigridPreconditioner(const MatrixFreeOperator<dim, fe_degree, operator_kind> &op,
                                   const AdditionalData &data = AdditionalData()) : op(op.handle()) {
    if (op.partitioned()) throw ExcMessage("MultigridPreconditioner: one block only (no multigrid across ranks)");
    bp5_mg_params_t prm{};
    prm.max_levels = (int32_t)data.max_levels;
    prm.smoothing_degree = (int32_t)data.degree;
    prm.smoothing_range = data.smoothing_range;
    prm.eig_iterations = (int32_t)data.eig_cg_n_iterations;
    prm.coarse_max_its = (int32_t)data.coarse_max_iterations;
    prm.coarse_tol = data.coarse_tolerance;
    check(bp5_mg_create(this->op, &prm, &h));
  }
  MultigridPreconditioner(const MultigridPreconditioner &) = delete;
  ~MultigridPreconditioner() { bp5_mg_destroy(h); }
  // PreconditionMG::vmult: dst = one V-cycle applied to src
  void vmult(VectorType &dst, const VectorType &src) const {
    check(bp5_mg_vcycle(h, dst.handle(), src.handle()));
    dst.mark_modified();
  }
  unsigned int n_levels() const { int n = 0; check(bp5_mg_n_levels(h, &n)); return (unsigned)n; }
  bp5_mg_t handle() const { return h; }
  bp5_operator_t operator_handle() const { return op; }

 private:
  bp5_operator_t op = nullptr;
  bp5_mg_t h = nullptr;
};
}  // namespace b200

// ------------------------------------------------------------------ solvers
namespace b200 {
// does MatrixType expose the library operator (BP5::PoissonOperator, Step64::HelmholtzOperator)?
template <typename M, typename = void> struct has_native_handle : std::false_type {};
template <typename M>
struct has_native_handle<M, std::void_t<decltype(std::declval<const M &>().handle()), decltype(std::declval<const M &>().do_zero_out),
                                        decltype(std::declval<const M &>().partitioned())>>
    : std::is_same<decltype(std::declval<const M &>().handle()), bp5_operator_t> {};

// a preconditioner with get_vector() is a DiagonalMatrix; any other one is applied through vmult(dst, src)
template <typename P, typename = void> struct has_get_vector : std::false_type {};
template <typename P>
struct has_get_vector<P, std::void_t<decltype(std::declval<const P &>().get_vector())>> : std::true_type {};
template <typename P> struct is_multigrid : std::false_type {};
template <int dim, int fe_degree, int kind>
struct is_multigrid<MultigridPreconditioner<dim, fe_degree, kind>> : std::true_type {};

template <typename VectorType, int variant> class SolverCGBase {
 public:
  explicit SolverCGBase(SolverControl &cn) : control(cn) {}
  virtual ~SolverCGBase() = default;

  template <typename MatrixType, typename PreconditionerType>
  void solve(const MatrixType &A, VectorType &x, const VectorType &b, const PreconditionerType &preconditioner) {
    if constexpr (has_get_vector<PreconditionerType>::value) {
      solve_diagonal(A, x, b, preconditioner);
    } else {
      static_assert(variant == BP5_CG_STANDARD,
                    "SolverCGFullMerge takes a DiagonalMatrix preconditioner only: use SolverCG with a multigrid or "
                    "other vmult preconditioner");
      if constexpr (has_native_handle<MatrixType>::value && is_multigrid<PreconditionerType>::value) {
        if (preconditioner.operator_handle() != A.handle())
          throw ExcMessage("SolverCG: the multigrid preconditioner was built on a different operator");
        // library operator + library multigrid: the whole loop is one native call
        int its = 0;
        double val = 0.0;
        const int rc = bp5_mg_cg_solve(preconditioner.handle(), x.handle(), b.handle(), control.abi_kind(),
                                       control.tolerance(), (int)control.max_steps(), &its, &val, nullptr, 0);
        if (rc == BP5_ERR_DIVIDE_BY_ZERO) { control.record((unsigned)its, val); throw ExcDivideByZero(); }
        finish(rc, its, val, x);
      } else {
        solve_standard_preconditioned(A, x, b, preconditioner);
      }
    }
  }

 protected:
  template <typename MatrixType, typename PreconditionerType>
  void solve_diagonal(const MatrixType &A, VectorType &x, const VectorType &b, const PreconditionerType &preconditioner) {
    // the reference passes a DiagonalMatrix of ones (bp5/step-64.cu:428-432) and reads it in every
    // pass; an all-ones diagonal is recognised and not read at all (SURVEY.md 8a, S4)
    const VectorType &diag = preconditioner.get_vector();
    bp5_vector_t dh = diag.is_constant_value(1.0) ? nullptr : diag.handle();
    if constexpr (has_native_handle<MatrixType>::value) {
      // library operator: the whole loop runs behind one ABI call with the tuned cell kernel
      int its = 0;
      double val = 0.0;
      if (A.partitioned()) {
        // one block per rank: the merged loop with its halo exchange and all-rank sums is one native call
        // (bp5_peer_cg_solve); "pcg-standard" runs the generic loop below around the partitioned vmult
        if constexpr (variant == BP5_CG_MERGED) {
          const int rc = bp5_peer_cg_solve(A.handle(), x.handle(), b.handle(), dh, control.abi_kind(), control.tolerance(),
                                           (int)control.max_steps(), &its, &val, nullptr, 0);
          finish(rc, its, val, x);
        } else {
          solve_standard_generic(A, x, b, diag, dh != nullptr);
        }
        return;
      }
      check(bp5_operator_set_zero_out(A.handle(), A.do_zero_out));
      const int rc = bp5_cg_solve(A.handle(), x.handle(), b.handle(), dh, variant, control.abi_kind(),
                                  control.tolerance(), (int)control.max_steps(), &its, &val, nullptr, 0);
      finish(rc, its, val, x);
    } else if constexpr (variant == BP5_CG_MERGED) {
      solve_merged_generic(A, x, b, dh);
    } else {
      solve_standard_generic(A, x, b, diag, dh != nullptr);
    }
  }

 protected:
  void finish(int rc, int its, double val, VectorType &x) {
    control.record((unsigned)its, val);
    x.mark_modified();
    if (rc == BP5_ERR_NO_CONVERGENCE) throw SolverControl::NoConvergence((unsigned)its, val);   // solver.h:539-540
    check(rc);
  }
  int host_check(unsigned step, double value) const {     // SolverControl::check [UPSTREAM]
    if (control.abi_kind() == BP5_CONTROL_ITERATION_NUMBER && step >= control.max_steps()) return 1;
    if (value <= control.tolerance()) return 1;
    if (step >= control.max_steps() || std::isnan(value)) return 2;
    return 0;
  }

  // SolverCGFullMerge::solve (bp5/solver.h:343-542) around ANY operator with vmult(dst, src) -- e.g. one
  // built from user-written device functors on CUDAWrappers::MatrixFree.  The update / dot-product kernels
  // and the scalar recurrences are the library's (stepwise ABI); A.vmult runs between them on the same
  // stream, so nothing but an "are we done" poll every few iterations reaches the host.
  template <typename MatrixType>
  void solve_merged_generic(const MatrixType &A, VectorType &x, const VectorType &b, bp5_vector_t dh) {
    bp5_operator_t op = bp5_vector_owner(x.handle());
    if (!op) throw ExcMessage("SolverCGFullMerge: x must come from initialize_dof_vector() or reinit(other)");
    VectorType g0;
    double res0;
    const bool x_zero = x.all_zero();                     // solver.h:375-381
    if (x_zero) res0 = b.l2_norm();
    else { g0.reinit(x); A.vmult(g0, x); g0.add(-1., b); res0 = g0.l2_norm(); }
    const int conv0 = host_check(0, res0);                // iteration_status(0, ...), solver.h:384
    if (conv0 != 0) { finish(conv0 == 2 ? BP5_ERR_NO_CONVERGENCE : BP5_OK, 0, res0, x); return; }
    check(bp5_cg_step_begin(op, x.handle(), b.handle(), dh, control.abi_kind(), control.tolerance(),
                            (int)control.max_steps(), res0, 0));
    bp5_vector_t gh, dd, hh;
    check(bp5_cg_step_vectors(op, &gh, &dd, &hh));
    if (!x_zero) check(bp5_vector_copy(gh, g0.handle()));
    VectorType d, h, sums;
    d.view(dd); h.view(hh);
    sums.reinit(8);
    int state = 0, its = 0;
    double val = res0;
    for (unsigned it = 1; it <= control.max_steps() && state == 0; ++it) {
      check(bp5_cg_step_update(op, (int)it));             // 1) solver.h:413-448 (also zeroes h)
      A.vmult(h, d);                                      // 2) solver.h:475
      check(bp5_cg_step_local_dots(op, sums.get_values()));   // 3) solver.h:478-485
      check(bp5_cg_step_scalars(op, sums.get_values()));      // 4) solver.h:497-533, on the device
      if (it % 8 == 0 || it == control.max_steps()) check(bp5_cg_step_poll(op, &state, &its, &val));
    }
    check(bp5_cg_step_finish(op, nullptr));               // owed x update, solver.h:509-526
    check(bp5_cg_step_poll(op, &state, &its, &val));
    if (state == 3) { control.record((unsigned)its, val); throw ExcDivideByZero(); }   // solver.h:501
    finish(state == 1 ? BP5_OK : BP5_ERR_NO_CONVERGENCE, its, val, x);
  }

  // dealii::SolverCG [UPSTREAM] with vector operations only ("pcg-standard", bp5/step-64.cu:446-453)
  template <typename MatrixType>
  void solve_standard_generic(const MatrixType &A, VectorType &x, const VectorType &b, const VectorType &diag,
                              bool has_diag) {
    VectorType g, d, h;
    g.reinit(x); d.reinit(x); h.reinit(x);
    if (!x.all_zero()) { A.vmult(g, x); g.add(-1., b); } else g.equ(-1., b);
    double res = g.l2_norm();
    unsigned it = 0;
    int conv = host_check(0, res);
    double gh = 0.;
    if (conv == 0) {
      if (has_diag) { h.equ(1., g); h.scale(diag); } else h.equ(1., g);
      d.equ(-1., h);
      gh = g * h;
    }
    while (conv == 0) {
      ++it;
      h = 0.;
      A.vmult(h, d);
      const double dAd = d * h;
      if (dAd == 0.) { control.record(it, res); throw ExcDivideByZero(); }
      const double alpha = gh / dAd;
      x.add(alpha, d);
      g.add(alpha, h);
      res = g.l2_norm();
      conv = host_check(it, res);
      if (conv != 0) break;
      if (has_diag) { h.equ(1., g); h.scale(diag); } else h.equ(1., g);
      const double gh_new = g * h;
      const double beta = gh_new / gh;
      gh = gh_new;
      d.sadd(beta, -1., h);
    }
    finish(conv == 2 ? BP5_ERR_NO_CONVERGENCE : BP5_OK, (int)it, res, x);
  }

  // dealii::SolverCG [UPSTREAM] around any operator and any preconditioner with vmult(dst, src)
  template <typename MatrixType, typename PreconditionerType>
  void solve_standard_preconditioned(const MatrixType &A, VectorType &x, const VectorType &b,
                                     const PreconditionerType &preconditioner) {
    VectorType g, d, h;
    g.reinit(x); d.reinit(x); h.reinit(x);
    if (!x.all_zero()) { A.vmult(g, x); g.add(-1., b); } else g.equ(-1., b);
    double res = g.l2_norm();
    unsigned it = 0;
    int conv = host_check(0, res);
    double gh = 0.;
    if (conv == 0) {
      preconditioner.vmult(h, g);
      d.equ(-1., h);
      gh = g * h;
    }
    while (conv == 0) {
      ++it;
      h = 0.;
      A.vmult(h, d);
      const double dAd = d * h;
      if (dAd == 0.) { control.record(it, res); throw ExcDivideByZero(); }
      const double alpha = gh / dAd;
      x.add(alpha, d);
      g.add(alpha, h);
      res = g.l2_norm();
      conv = host_check(it, res);
      if (conv != 0) break;
      preconditioner.vmult(h, g);
      const double gh_new = g * h;
      const double beta = gh_new / gh;
      gh = gh_new;
      d.sadd(beta, -1., h);
    }
    finish(conv == 2 ? BP5_ERR_NO_CONVERGENCE : BP5_OK, (int)it, res, x);
  }

  SolverControl &control;
};
}  // namespace b200

// dealii::SolverCG as the drivers use it ("pcg-standard", bp5/step-64.cu:446-453)
template <typename VectorType> class SolverCG : public b200::SolverCGBase<VectorType, BP5_CG_STANDARD> {
 public:
  using b200::SolverCGBase<VectorType, BP5_CG_STANDARD>::SolverCGBase;
};
// SolverCGFullMerge (bp5/solver.h:15-31), "pcg-merged"
template <typename VectorType> class SolverCGFullMerge : public b200::SolverCGBase<VectorType, BP5_CG_MERGED> {
 public:
  using b200::SolverCGBase<VectorType, BP5_CG_MERGED>::SolverCGBase;
};

// ------------------------------------------------------------------ small utilities of the drivers
class Timer {
 public:
  Timer() : t0(std::chrono::steady_clock::now()) {}
  double wall_time() const { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); }

 private:
  std::chrono::steady_clock::time_point t0;
};

class ConditionalOStream {
 public:
  ConditionalOStream(std::ostream &os, bool active) : os(os), active(active) {}
  template <typename T> const ConditionalOStream &operator<<(const T &t) const { if (active) os << t; return *this; }
  const ConditionalOStream &operator<<(std::ostream &(*f)(std::ostream &)) const { if (active) os << f; return *this; }

 private:
  std::ostream &os;
  bool active;
};

}  // namespace dealii

// ------------------------------------------------------------------ the two operators of the reference
namespace BP5 {
// quadrature: BP5_QUAD_GAUSS is the reference default, BP5_QUAD_GLL its COLLOCATION switch (bp5/step-64.cu:48,243-247)
template <int dim, int fe_degree>
class PoissonOperator : public dealii::b200::MatrixFreeOperator<dim, fe_degree, BP5_OP_POISSON> {
 public:
  PoissonOperator(const dealii::DoFHandler<dim> &dof_handler, const dealii::AffineConstraints<double> &constraints,
                  int quadrature = BP5_QUAD_GAUSS, bool use_coloring = false)
      : dealii::b200::MatrixFreeOperator<dim, fe_degree, BP5_OP_POISSON>(dof_handler, constraints, quadrature,
                                                                         use_coloring) {}
};
}  // namespace BP5

namespace Step64 {
template <int dim, int fe_degree>
class HelmholtzOperator : public dealii::b200::MatrixFreeOperator<dim, fe_degree, BP5_OP_HELMHOLTZ> {
 public:
  HelmholtzOperator(const dealii::DoFHandler<dim> &dof_handler, const dealii::AffineConstraints<double> &constraints)
      : dealii::b200::MatrixFreeOperator<dim, fe_degree, BP5_OP_HELMHOLTZ>(dof_handler, constraints, BP5_QUAD_GAUSS) {
    this->do_zero_out = true;                                       // step-64/step-64.cu:316 (dst = 0.)
  }
};
}  // namespace Step64
