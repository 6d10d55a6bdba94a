// Host side of the cell loop: kernel selection per (degree, quadrature,
// operator), persistent-grid sizing, skeleton zeroing and the Dirichlet copy
// (MatrixFree::cell_loop / copy_constrained_values, bp5/step-64.cu:274-275).
#include "apply_launch.cuh"

namespace bp5 {

static int cells_per_tile_for(int p) {
  switch (p) {
    case 1: return TileCells<1>::value; case 2: return TileCells<2>::value;
    case 3: return TileCells<3>::value; case 4: return TileCells<4>::value;
    case 5: return TileCells<5>::value; case 6: return TileCells<6>::value;
    case 7: return TileCells<7>::value; case 8: return TileCells<8>::value;
  }
  return 0;
}

int apply_choose(bp5_operator_t op) {
  int cpt = cells_per_tile_for(op->p);
  BP5_REQUIRE(cpt > 0, "degree must be 1..8");
  if (op->prob.geometry_mode == BP5_GEOM_ON_THE_FLY) {
    // collocation + Poisson: the four-fields-at-once kernel (apply_otf.cuh) up to p = 4, the general kernel above
    // (p = 5: 21.9 against 19.9, p = 6: 23.3 against 20.9 GDoF/s per vmult on a deformed mesh)
    op->otf_general = !(op->prob.quadrature == BP5_QUAD_GLL && op->prob.operator_kind == BP5_OP_POISSON) || op->p >= 5;
#ifdef BP5_TUNING_ENV        // tuning builds only
    if (const char *v = getenv("BP5_OTF_GENERAL"))   // 0 / 1: which kernel takes collocation + Poisson
      op->otf_general = atoi(v) != 0 || !(op->prob.quadrature == BP5_QUAD_GLL && op->prob.operator_kind == BP5_OP_POISSON);
#endif
    switch (op->p) {
#define BP5_OTF_CASE(P) case P: cpt = op->otf_general ? OtfgTileCells<P>::value : OtfTileCells<P>::value; break;
      BP5_OTF_CASE(1) BP5_OTF_CASE(2) BP5_OTF_CASE(3) BP5_OTF_CASE(4) BP5_OTF_CASE(5) BP5_OTF_CASE(6) BP5_OTF_CASE(7) BP5_OTF_CASE(8)
#undef BP5_OTF_CASE
    }
  }
  const int n3 = op->n * op->n * op->n;
  op->cells_per_tile = cpt;
  operator_plan_tiles(op);
  op->tile_doubles = ((int64_t)cpt * op->metric_planes * n3 + 1) & ~(int64_t)1;
  // how the metric reaches the quadrature phase (ApplyCfg::MLOAD); BP5_MLOAD overrides for tuning runs
  op->metric_path = 0;
  // geometry on the fly on an undeformed (axis-parallel) mesh: one constant Jacobian, no coordinate gathers
  const bool otf_affine = op->prob.geometry_mode == BP5_GEOM_ON_THE_FLY && op->prob.deformation == 0 &&
                          op->prob.operator_kind == BP5_OP_POISSON;
  if (otf_affine) { op->metric_path = 3; cpt = cells_per_tile_for(op->p); op->cells_per_tile = cpt; operator_plan_tiles(op); }
#ifdef BP5_ENABLE_MLOAD
  if (const char *mv = getenv("BP5_MLOAD")) op->metric_path = atoi(mv);
#endif
  BP5_REQUIRE(op->metric_path >= 0 && op->metric_path <= 3, "BP5_MLOAD must be 0, 1 or 2");
  static const char *const kPath[4] = {"metric=tma-smem", "metric=ldg-regs", "metric=ldg-regs-ahead",
                                       "geometry=on-the-fly(affine: constant Jacobian)"};
  char name[160];
  snprintf(name, sizeof(name), "bp5_apply_kernel<p=%d,%s,%s,cells_per_tile=%d,%s>", op->p,
           op->prob.quadrature == BP5_QUAD_GLL ? "gll-collocation" : "gauss",
           op->prob.operator_kind == BP5_OP_HELMHOLTZ ? "helmholtz" : "poisson", cpt, kPath[op->metric_path]);
  if (op->prob.geometry_mode == BP5_GEOM_ON_THE_FLY && !otf_affine) {
    const bool special = !op->otf_general;
    snprintf(name, sizeof(name), "%s<p=%d,%s,%s,cells_per_tile=%d,geometry=on-the-fly>",
             special ? "bp5_apply_otf_kernel" : "bp5_apply_otfg_kernel", op->p,
             op->prob.quadrature == BP5_QUAD_GLL ? "gll-collocation" : "gauss",
             op->prob.operator_kind == BP5_OP_HELMHOLTZ ? "helmholtz" : "poisson", cpt);
  }
  op->kernel_name = name;
  return BP5_OK;
}

// mode: 0 dst += A src ; 1 overwrite cell-interior DoFs ; 2 = 1 + per-CTA partial sums of src . (A src)
template <int P, int MLOAD>
static int launch_pm(bp5_operator_t op, double *dst, const double *src, int mode, double *dp, int which) {
  const bool gll = op->prob.quadrature == BP5_QUAD_GLL;
  const bool helm = op->prob.operator_kind == BP5_OP_HELMHOLTZ;
#define BP5_LAUNCH_MODE(M)                                                                                       \
  (gll ? (helm ? launch<P, 1, 1, M, MLOAD>(op, dst, src, dp, which) : launch<P, 1, 0, M, MLOAD>(op, dst, src, dp, which))      \
       : (helm ? launch<P, 0, 1, M, MLOAD>(op, dst, src, dp, which) : launch<P, 0, 0, M, MLOAD>(op, dst, src, dp, which)))
  if constexpr (MLOAD == 0) {
    if (op->hanging) return launch_hanging(op, dst, src, mode, dp, which);   // hanging-node constraints (apply_hang.cu)
    if (mode >= 3) return launch_colored(op, dst, src, mode, dp, which);     // one colour, plain adds (apply_colored.cu)
  }
  if (mode == 2) return BP5_LAUNCH_MODE(2);
  if (mode == 1) return BP5_LAUNCH_MODE(1);
  return BP5_LAUNCH_MODE(0);
#undef BP5_LAUNCH_MODE
}

// geometry on the fly, affine mesh (MLOAD = 3): Poisson only
template <int P>
static int launch_affine(bp5_operator_t op, double *dst, const double *src, int mode, double *dp, int which) {
  const bool gll = op->prob.quadrature == BP5_QUAD_GLL;
#define BP5_LAUNCH_AFF(M) (gll ? launch<P, 1, 0, M, 3>(op, dst, src, dp, which) : launch<P, 0, 0, M, 3>(op, dst, src, dp, which))
  if (mode == 2) return BP5_LAUNCH_AFF(2);
  if (mode == 1) return BP5_LAUNCH_AFF(1);
  return BP5_LAUNCH_AFF(0);
#undef BP5_LAUNCH_AFF
}

template <int P>
static int launch_p(bp5_operator_t op, double *dst, const double *src, int mode, double *dp, int which) {
  if (op->metric_path == 3) return launch_affine<P>(op, dst, src, mode, dp, which);
#ifdef BP5_ENABLE_MLOAD   // tuning builds: metric straight to registers (measured slower, profiles/r1_v3_notes.md)
  if (op->metric_path == 1) return launch_pm<P, 1>(op, dst, src, mode, dp, which);
  if (op->metric_path == 2) return launch_pm<P, 2>(op, dst, src, mode, dp, which);
#endif
  return launch_pm<P, 0>(op, dst, src, mode, dp, which);
}

// overwrite_interior: dst's skeleton (shared DoFs, see zero_skeleton) must be
// zero on entry, cell-interior DoFs are overwritten; otherwise dst += A src.
// dot_partials != nullptr (needs overwrite_interior): the kernel also leaves op->apply_grid per-CTA parts of
// src . (A src) there (see bp5_apply_kernel, OVERWRITE == 2).
static int apply_dispatch(bp5_operator_t op, double *dst, const double *src, int mode, double *dot_partials, int which) {
  if (op->prob.geometry_mode == BP5_GEOM_ON_THE_FLY && op->metric_path != 3)
    return apply_cell_loop_otfg(op, dst, src, mode, dot_partials, which);
  switch (op->p) {
    case 1: return launch_p<1>(op, dst, src, mode, dot_partials, which);
    case 2: return launch_p<2>(op, dst, src, mode, dot_partials, which);
    case 3: return launch_p<3>(op, dst, src, mode, dot_partials, which);
    case 4: return launch_p<4>(op, dst, src, mode, dot_partials, which);
    case 5: return launch_p<5>(op, dst, src, mode, dot_partials, which);
    case 6: return launch_p<6>(op, dst, src, mode, dot_partials, which);
    case 7: return launch_p<7>(op, dst, src, mode, dot_partials, which);
    case 8: return launch_p<8>(op, dst, src, mode, dot_partials, which);
  }
  set_error("unsupported degree %d", op->p);
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

int apply_copy_constrained_dot(bp5_operator_t op, double *dst, const double *src, double *partials) {
  copy_constrained_dot_kernel<<<kConstrainedPartials, 256, 0, op->ctx->stream>>>(op->constrained, op->n_constrained, src,
                                                                                dst, partials);
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
