// The merged CG's cell loop in the blocked layout (bp5_apply_kernel with BLK): a separate file only to compile in
// parallel.
#include "apply_launch.cuh"

namespace bp5 {

int apply_blocked_kernel_resources(bp5_operator_t op, int *ctas, size_t *local) {
  return op_cg_kernel_resources<true>(op, ctas, local);
}

int apply_cell_loop_blocked(bp5_operator_t op, double *dst, const double *src, double *dot_partials) {
  BP5_REQUIRE(op->blk_desc != nullptr && dot_partials != nullptr, "blocked cell loop without its layout or partials");
  if (op->cell_kernel == CellKernel::kAffine)   // Poisson only
    return with_degree(op->p, [&](auto P) {
      return with_value<0, 1>(op->prob.quadrature == BP5_QUAD_GLL, [&](auto quad) {
        return launch<P, quad, 0, 2, true, 0, true>(op, dst, src, dot_partials, 0);
      });
    });
  BP5_REQUIRE(op->cell_kernel == CellKernel::kStored && !op->hanging, "the blocked layout has no kernel for this operator");
  return with_degree(op->p, [&](auto P) {
    return with_quad_op(op, [&](auto quad, auto helm) {
      return launch<P, quad, helm, 2, false, 0, true>(op, dst, src, dot_partials, 0);
    });
  });
}

}  // namespace bp5
