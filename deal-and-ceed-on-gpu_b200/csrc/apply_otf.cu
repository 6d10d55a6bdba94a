// Host side of the on-the-fly-geometry cell kernel (apply_otf.cuh): launch per degree and mode.
#include "apply_launch.cuh"
#include "apply_otf.cuh"

namespace bp5 {

int apply_cell_loop_otf(bp5_operator_t op, double *dst, const double *src, int mode, double *dot_partials, int which) {
  return with_degree(op->p, [&](auto P) {
    return with_value<0, 1, 2>(mode, [&](auto m) {
      constexpr int CPT = OtfTileCells<P>::value;
      using Cfg = ApplyOtfCfg<P, CPT>;
      ApplyOtfParams<P + 1> prm;
      fill_common_params<P + 1>(prm, op, dst, src, dot_partials, which);
      const long long n_local = op->n_owned + op->n_ghost;
      prm.cx = op->coords; prm.cy = op->coords + n_local; prm.cz = op->coords + 2 * n_local;
      return launch_cell_kernel<bp5_apply_otf_kernel<P, CPT, m>>(op, prm, Cfg::NT, Cfg::SMEM_BYTES,
                                                                   cudaSharedmemCarveoutDefault);
    });
  });
}

}  // namespace bp5
