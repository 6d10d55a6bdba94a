// Host side of the cell loop: kernel selection per (degree, quadrature,
// operator), persistent-grid sizing, skeleton zeroing and the Dirichlet copy
// (MatrixFree::cell_loop / copy_constrained_values, bp5/step-64.cu:274-275).
#include "apply_launch.cuh"

namespace bp5 {

int apply_choose(bp5_operator_t op) {
  const bool gll = op->prob.quadrature == BP5_QUAD_GLL, helm = op->prob.operator_kind == BP5_OP_HELMHOLTZ;
  if (op->prob.geometry_mode != BP5_GEOM_ON_THE_FLY)
    op->cell_kernel = CellKernel::kStored;
  else if (op->prob.deformation == 0 && !helm)   // undeformed (axis-parallel) mesh: no coordinate gathers
    op->cell_kernel = CellKernel::kAffine;
  else if (gll && !helm && op->p <= 4)
    // collocation + Poisson: the four-fields-at-once kernel (apply_otf.cuh) up to p = 4, the general kernel above
    // (p = 5: 21.9 against 19.9, p = 6: 23.3 against 20.9 GDoF/s per vmult on a deformed mesh)
    op->cell_kernel = CellKernel::kOnTheFly;
  else
    op->cell_kernel = CellKernel::kOnTheFlyGeneral;
  int cpt = 0;
  const int rc = with_degree(op->p, [&](auto P) {
    constexpr int p = decltype(P)::value;
    cpt = op->cell_kernel == CellKernel::kOnTheFly          ? OtfTileCells<p>::value
          : op->cell_kernel == CellKernel::kOnTheFlyGeneral ? OtfgTileCells<p>::value
                                                            : TileCells<p>::value;
    return BP5_OK;
  });
  if (rc != BP5_OK) return rc;
  op->cells_per_tile = cpt;
  operator_plan_tiles(op);
  const int n3 = op->n * op->n * op->n;
  op->tile_doubles = ((int64_t)cpt * op->metric_planes * n3 + 1) & ~(int64_t)1;
  const char *quad = gll ? "gll-collocation" : "gauss", *kind = helm ? "helmholtz" : "poisson";
  char name[160];
  if (op->cell_kernel == CellKernel::kStored || op->cell_kernel == CellKernel::kAffine)
    snprintf(name, sizeof(name), "bp5_apply_kernel<p=%d,%s,%s,cells_per_tile=%d,%s>", op->p, quad, kind, cpt,
             op->cell_kernel == CellKernel::kAffine ? "geometry=on-the-fly(affine: constant Jacobian)" : "metric=tma-smem");
  else
    snprintf(name, sizeof(name), "%s<p=%d,%s,%s,cells_per_tile=%d,geometry=on-the-fly>",
             op->cell_kernel == CellKernel::kOnTheFly ? "bp5_apply_otf_kernel" : "bp5_apply_otfg_kernel", op->p, quad,
             kind, cpt);
  op->kernel_name = name;
  return BP5_OK;
}

// mode: 0 dst += A src ; 1 overwrite cell-interior DoFs ; 2 = 1 + per-CTA partial sums of src . (A src) ;
// 3..5 the same for one colour of the coloured cell order (plain adds)
// overwrite_interior: dst's skeleton (shared DoFs, see zero_skeleton) must be
// zero on entry, cell-interior DoFs are overwritten; otherwise dst += A src.
// dot_partials != nullptr (needs overwrite_interior): the kernel also leaves op->apply_grid per-CTA parts of
// src . (A src) there (see bp5_apply_kernel, OVERWRITE == 2).
static int apply_dispatch(bp5_operator_t op, double *dst, const double *src, int mode, double *dp, int which) {
  switch (op->cell_kernel) {
    case CellKernel::kOnTheFly: return apply_cell_loop_otf(op, dst, src, mode, dp, which);
    case CellKernel::kOnTheFlyGeneral: return apply_cell_loop_otfg(op, dst, src, mode, dp, which);
    case CellKernel::kAffine:   // Poisson only
      return with_degree(op->p, [&](auto P) {
        return with_value<0, 1>(op->prob.quadrature == BP5_QUAD_GLL, [&](auto quad) {
          return with_value<0, 1, 2>(mode, [&](auto m) {
            return launch<P, quad, 0, m, true>(op, dst, src, dp, which);
          });
        });
      });
    case CellKernel::kStored:
      if (op->hanging) return launch_hanging(op, dst, src, mode, dp, which);   // hanging-node constraints (apply_hang.cu)
      if (mode >= 3) return launch_colored(op, dst, src, mode, dp, which);     // one colour, plain adds (apply_colored.cu)
      return with_degree(op->p, [&](auto P) {
        return with_quad_op(op, [&](auto quad, auto helm) {
          return with_value<0, 1, 2>(mode, [&](auto m) { return launch<P, quad, helm, m>(op, dst, src, dp, which); });
        });
      });
  }
  set_error("unknown cell kernel");
  return BP5_ERR_UNSUPPORTED;
}

int apply_cell_loop(bp5_operator_t op, double *dst, const double *src, bool overwrite_interior, double *dot_partials,
                    int which) {
  BP5_REQUIRE(dot_partials == nullptr || overwrite_interior, "the fused dot product needs the overwrite kernel");
  const int mode = dot_partials ? 2 : (overwrite_interior ? 1 : 0);
  if (op->hanging) {
    // locally refined mesh: the tiles with constrained / table cells through the kernel with the constraint exchange,
    // then all others; the per-CTA partial sums of the fused dot product one group after the other
    BP5_REQUIRE(op->range_begin < 0 && which == 0, "locally refined meshes run whole cell loops only");
    int rc = apply_dispatch(op, dst, src, mode, dot_partials, 1);
    const int first = op->apply_grid;
    if (rc == BP5_OK) rc = apply_dispatch(op, dst, src, mode, dot_partials ? dot_partials + first : nullptr, 2);
    op->apply_grid += first;
    return rc;
  }
  if (op->prob.cell_order != BP5_CELL_ORDER_COLORED) return apply_dispatch(op, dst, src, mode, dot_partials, which);
  // coloured cell order: one launch per colour over that colour's tiles, in a fixed order on one stream; the
  // per-CTA partial sums of the fused dot product are laid out colour after colour.
  BP5_REQUIRE(op->range_begin < 0 && which == 0, "the coloured cell order runs whole cell loops only");
  int total = 0, rc = BP5_OK;
  op->grid_cap = kApplyPartialCap / 8;
  for (int c = 0; c < 8 && rc == BP5_OK; ++c) {
    op->range_begin = op->color_tile_begin[c];
    op->range_end = op->color_tile_begin[c + 1];
    rc = apply_dispatch(op, dst, src, mode + 3, dot_partials ? dot_partials + total : nullptr, 0);
    total += op->apply_grid;
  }
  op->range_begin = -1; op->range_end = -1;
  op->grid_cap = 0;
  op->apply_grid = total;
  return rc;
}

// the lexicographic in-loop kernels live in this file, the blocked ones in apply_blocked.cu
int apply_cg_kernel_resources(bp5_operator_t op, bool blocked, int *ctas, size_t *local) {
  if (blocked) return apply_blocked_kernel_resources(op, ctas, local);
  return op_cg_kernel_resources<false>(op, ctas, local);
}

// "dst = 0" (bp5/step-64.cu:270-271) only has to reach the skeleton -- DoFs shared by several cells and the
// ghosts; cell-interior DoFs are stored by the OVERWRITE kernel.  Measured (profiles/r1_v2_notes.md): zeroing
// only the skeleton through a bit mask is SLOWER than a full memset (scattered partial-sector writes) and saves
// no DRAM traffic, because L2 fills partially written sectors anyway.  So it is a plain memset.
int apply_zero_skeleton(bp5_operator_t op, double *dst) {
  BP5_CUDA(cudaMemsetAsync(dst, 0, sizeof(double) * (op->n_owned + op->n_ghost), op->ctx->stream));
  return BP5_OK;
}

// copy_constrained_values [UPSTREAM], called at bp5/step-64.cu:275:
// dst[c] = src[c] on Dirichlet dofs.
__global__ void copy_constrained_kernel(const int *__restrict__ list, long long n, const double *__restrict__ src,
                                        double *__restrict__ dst) {
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (t < n) { const int i = list[t]; dst[i] = src[i]; }
}

// The same copy, and the correction the fused dot product needs: the cell kernel summed src_c * (A src)_c
// for the Dirichlet rows too, but dst_c becomes src_c, so add sum_c src_c * (src_c - (A src)_c).  Exactly
// zero whenever src vanishes on the Dirichlet set (always, inside the reference's CG).  Fixed grid,
// per-block partials: deterministic.
__global__ void __launch_bounds__(256) copy_constrained_dot_kernel(const int *__restrict__ list, long long n,
                                                                   const double *__restrict__ src,
                                                                   double *__restrict__ dst,
                                                                   double *__restrict__ partials) {
  __shared__ double sh[8];
  double acc = 0.0;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
    const int i = list[t];
    const double s = src[i];
    acc += s * (s - dst[i]);
    dst[i] = s;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = threadIdx.x < 8 ? sh[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (threadIdx.x == 0) partials[blockIdx.x] = acc;
  }
}

int apply_copy_constrained_dot(bp5_operator_t op, const int *list, double *dst, const double *src, double *partials) {
  copy_constrained_dot_kernel<<<kConstrainedPartials, 256, 0, op->ctx->stream>>>(list, op->n_constrained, src, dst,
                                                                                partials);
  BP5_CHECK_LAUNCH();
  op->ctx->launches++;
  return BP5_OK;
}

int apply_copy_constrained(bp5_operator_t op, double *dst, const double *src) {
  if (op->n_constrained == 0) return BP5_OK;
  const long long n = op->n_constrained;
  copy_constrained_kernel<<<(unsigned)((n + 255) / 256), 256, 0, op->ctx->stream>>>(op->constrained, n, src, dst);
  BP5_CHECK_LAUNCH();
  op->ctx->launches++;
  return BP5_OK;
}

}  // namespace bp5
