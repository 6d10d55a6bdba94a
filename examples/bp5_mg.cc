// BP5 (Poisson) and step-64 (variable-coefficient Helmholtz) solved to 1e-10 |b| with SolverCG, once with the
// Jacobi preconditioner (DiagonalMatrix of the inverse diagonal) and once with the geometric multigrid V-cycle
// (b200::MultigridPreconditioner: Chebyshev-Jacobi smoothing, CG on the coarsest level).  Prints the iterations,
// ||u||_L2 and the solve time of each.
//   bp5_mg [--degree p] [--cells c] [--problem bp5|helmholtz|both]
#include <cstdlib>
#include <cstring>
#include <iomanip>
#include <string>

#include "dealii_b200/dealii_b200.h"

using namespace dealii;
using VectorType = LinearAlgebra::distributed::Vector<double, MemorySpace::CUDA>;

template <typename Operator> void solve_both(const char *name, const DoFHandler<3> &dof_handler, Operator &A) {
  VectorType x, b;
  A.initialize_dof_vector(x);
  b.reinit(x);
  A.assemble_rhs(b);
  const double tol = 1e-10 * b.l2_norm();
  std::cout << name << ": " << dof_handler.n_dofs() << " DoFs" << std::endl;
  {
    DiagonalMatrix<VectorType> jacobi;
    jacobi.get_vector().reinit(x);
    A.compute_inverse_diagonal(jacobi.get_vector());
    SolverControl control(100000, tol);
    x = 0.;
    Timer timer;
    SolverCG<VectorType>(control).solve(A, x, b, jacobi);
    const double t = timer.wall_time();
    std::cout << "  jacobi: Solved in " << control.last_step() << " iterations, time " << t << " s, solution norm: "
              << A.l2_norm(x) << std::endl;
  }
  {
    Timer setup;
    b200::MultigridPreconditioner<3, Operator::degree, Operator::kind> mg(A);
    const double ts = setup.wall_time();
    SolverControl control(100, tol);
    x = 0.;
    Timer timer;
    SolverCG<VectorType>(control).solve(A, x, b, mg);
    const double t = timer.wall_time();
    std::cout << "  multigrid (" << mg.n_levels() << " levels, set-up " << ts << " s): Solved in "
              << control.last_step() << " iterations, time " << t << " s, solution norm: " << A.l2_norm(x) << std::endl;
  }
}

template <int p> struct BP5Op : BP5::PoissonOperator<3, p> {
  static constexpr int degree = p, kind = BP5_OP_POISSON;
  using BP5::PoissonOperator<3, p>::PoissonOperator;
};
template <int p> struct HelmholtzOp : Step64::HelmholtzOperator<3, p> {
  static constexpr int degree = p, kind = BP5_OP_HELMHOLTZ;
  using Step64::HelmholtzOperator<3, p>::HelmholtzOperator;
};

template <int p> void run(unsigned cells, const std::string &problem) {
  Triangulation<3> triangulation;
  Point<3> upper;
  for (int d = 0; d < 3; ++d) upper[d] = 1.;
  GridGenerator::subdivided_hyper_rectangle(triangulation, std::vector<unsigned int>(3, cells), Point<3>(), upper);
  FE_Q<3> fe(p);
  DoFHandler<3> dof_handler(triangulation);
  dof_handler.distribute_dofs(fe);
  AffineConstraints<double> constraints;
  if (problem == "bp5" || problem == "both") {
    BP5Op<p> A(dof_handler, constraints);
    solve_both("BP5", dof_handler, A);
  }
  if (problem == "helmholtz" || problem == "both") {
    HelmholtzOp<p> A(dof_handler, constraints);
    solve_both("step-64 Helmholtz", dof_handler, A);
  }
}

int main(int argc, char *argv[]) {
  int degree = 4;
  unsigned cells = 16;
  std::string problem = "both";
  for (int i = 1; i + 1 < argc; i += 2) {
    if (!std::strcmp(argv[i], "--degree")) degree = std::atoi(argv[i + 1]);
    else if (!std::strcmp(argv[i], "--cells")) cells = (unsigned)std::atoi(argv[i + 1]);
    else if (!std::strcmp(argv[i], "--problem")) problem = argv[i + 1];
    else { std::cerr << "unknown argument " << argv[i] << std::endl; return 2; }
  }
  std::cout << std::setprecision(12);
  try {
    switch (degree) {
      case 2: run<2>(cells, problem); break;
      case 3: run<3>(cells, problem); break;
      case 4: run<4>(cells, problem); break;
      case 6: run<6>(cells, problem); break;
      default: std::cerr << "degree must be 2, 3, 4 or 6" << std::endl; return 2;
    }
  } catch (std::exception &exc) {
    std::cerr << "Exception on processing: " << std::endl << exc.what() << std::endl << "Aborting!" << std::endl;
    return 1;
  }
  return 0;
}
