// Instantiations of the cell kernel for locally refined meshes (apply.cuh): HANG = 1 resolves hanging-node constraints
// (the first tile group), HANG = 2 only knows the stride classes of the refined numbering (all other tiles).  A separate translation unit only so that it compiles in parallel with apply.cu.
#include "apply_launch.cuh"

namespace bp5 {

int launch_hanging(bp5_operator_t op, double *dst, const double *src, int mode, double *dp, int which) {
  BP5_REQUIRE(mode >= 0 && mode <= 2, "the coloured cell order is not available on locally refined meshes");
  BP5_REQUIRE(which == 1 || which == 2, "launch_hanging: one of the two tile groups at a time");
  // which == 1: tiles [0, n_boundary_tiles), constrained cells and cells with an index table
  return with_degree(op->p, [&](auto P) {
    return with_quad_op(op, [&](auto quad, auto helm) {
      return with_value<0, 1, 2>(mode, [&](auto m) {
        return with_value<1, 2>(which, [&](auto hang) {
          return launch<P, quad, helm, m, false, hang>(op, dst, src, dp, which);
        });
      });
    });
  });
}

}  // namespace bp5
