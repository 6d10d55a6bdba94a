// Instantiations of the cell kernel for the coloured cell order (OWMODE 3..5: plain adds, one colour per launch;
// apply.cuh).  A separate translation unit only so that it compiles in parallel with apply.cu.
#include "apply_launch.cuh"

namespace bp5 {

int launch_colored(bp5_operator_t op, double *dst, const double *src, int mode, double *dp, int which) {
  BP5_REQUIRE(mode >= 3 && mode <= 5, "launch_colored: mode must be 3..5");
  return with_degree(op->p, [&](auto P) {
    return with_quad_op(op, [&](auto quad, auto helm) {
      return with_value<3, 4, 5>(mode, [&](auto m) { return launch<P, quad, helm, m>(op, dst, src, dp, which); });
    });
  });
}

}  // namespace bp5
