// Device-resident state of a CG solve and the scalar recurrences of SolverCGFullMerge (bp5/solver.h:497-533),
// shared by the stand-alone CG kernels (cg.cu) and the fused per-iteration kernel (fused.cuh).
#pragma once
#include "common.h"

namespace bp5 {

struct CgState {
  double alpha, beta, alpha_old, beta_old;
  double res, tol, gh;
  int it;          // iterations completed == SolverControl::last_step()
  int state;       // 0 iterate, 1 success, 2 failure (max its / nan), 3 divide by zero
  int max_its, control;
  unsigned ticket;
  int history_len;
};

// SolverControl::check / IterationNumberControl::check [UPSTREAM]
__host__ __device__ __forceinline__ int control_check(int control, int step, int max_its, double value, double tol) {
  if (control == BP5_CONTROL_ITERATION_NUMBER && step >= max_its) return 1;
  if (value <= tol) return 1;
  if (step >= max_its || isnan(value)) return 2;
  return 0;
}

// scalar recurrences of one iteration from the seven (globally summed) dot products
// (solver.h:497-533); one thread
__device__ __forceinline__ void cg_scalar_step(CgState *st, const double (&rr)[7], double *history) {
  const int it = st->it + 1;
  st->alpha_old = st->alpha;
  st->beta_old = st->beta;
  st->it = it;
  if (rr[0] == 0.0) { st->state = 3; return; }                 // ExcDivideByZero, solver.h:501
  const double alpha = rr[6] / rr[0];                         // solver.h:502
  // solver.h:504-505; finite negatives are clamped at 0 (deviation): at exact convergence the
  // three-term expression can round slightly negative and the unguarded sqrt would report NaN.
  // A NaN expression (overflow, indefinite operator, inf in diag) must stay NaN so that the
  // stopping test fails like the reference's (fmax(0, NaN) would turn it into "converged").
  const double res_sq = rr[3] + 2 * alpha * rr[2] + alpha * alpha * rr[1];
  const double res = (res_sq < 0.0) ? 0.0 : sqrt(res_sq);
  st->alpha = alpha;
  st->res = res;
  if (history && it < st->history_len) history[it] = res;
  const int conv = control_check(st->control, it, st->max_its, res, st->tol);
  if (conv != 0) { st->state = conv; return; }
  st->beta = alpha * (rr[4] + alpha * rr[5]) / rr[6];         // solver.h:533
}

}  // namespace bp5
