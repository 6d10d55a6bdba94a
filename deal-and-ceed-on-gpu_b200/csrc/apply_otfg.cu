// Host side of the general on-the-fly-geometry cell kernel (apply_otfg.cuh): launch per degree, quadrature,
// operator and mode.  Gauss-Lobatto collocation + Poisson keeps its specialised kernel up to p = 4 (apply_otf.cu).
#include "apply_launch.cuh"
#include "apply_otfg.cuh"

namespace bp5 {

int apply_cell_loop_otfg(bp5_operator_t op, double *dst, const double *src, int mode, double *dot_partials, int which) {
  return with_degree(op->p, [&](auto P) {
    return with_quad_op(op, [&](auto quad, auto helm) {
      return with_value<0, 1, 2>(mode, [&](auto m) {
        constexpr int CPT = OtfgTileCells<P>::value;
        using Cfg = ApplyOtfgCfg<P, helm, CPT>;
        ApplyOtfgParams<P + 1> prm;
        fill_common_params<P + 1>(prm, op, dst, src, dot_partials, which);
        const long long n_local = op->n_owned + op->n_ghost;
        prm.cx = op->coords; prm.cy = op->coords + n_local; prm.cz = op->coords + 2 * n_local;
        return launch_cell_kernel<bp5_apply_otfg_kernel<P, quad, helm, CPT, m>>(op, prm, Cfg::NT, Cfg::SMEM_BYTES,
                                                                                 cudaSharedmemCarveoutDefault);
      });
    });
  });
}

}  // namespace bp5
