// Host-side launch of the cell kernels: the compile-time dispatch over degree, quadrature, operator and mode, the
// parameter fields all kernels share, and one launch path (persistent grid sizing, profiling events).  Shared by the
// translation units that hold the instantiations -- apply.cu (stored metric, affine), apply_colored.cu (plain adds for
// the coloured cell order), apply_hang.cu (hanging-node constraints), apply_otf.cu and apply_otfg.cu (geometry on the
// fly) -- which are separate files only to compile in parallel.
#pragma once
#include <type_traits>

#include "apply.cuh"
#include "tile_cells.h"

namespace bp5 {

// f(std::integral_constant<int, V>{}) for the V among Vs that equals v
template <int... Vs, class F>
static int with_value(int v, F &&f) {
  int rc = BP5_ERR_UNSUPPORTED;
  if (!((v == Vs && (rc = f(std::integral_constant<int, Vs>{}), true)) || ...)) set_error("unsupported case %d", v);
  return rc;
}
template <class F>
static int with_degree(int p, F &&f) { return with_value<1, 2, 3, 4, 5, 6, 7, 8>(p, f); }

// f(QUAD, HELM) as integral constants: QUAD 1 = Gauss-Lobatto collocation, HELM 1 = Helmholtz
template <class F>
static int with_quad_op(bp5_operator_t op, F &&f) {
  return with_value<0, 1>(op->prob.quadrature == BP5_QUAD_GLL, [&](auto quad) {
    return with_value<0, 1>(op->prob.operator_kind == BP5_OP_HELMHOLTZ, [&](auto helm) { return f(quad, helm); });
  });
}

// The fields every cell kernel's parameter struct has under the same names.  which: 0 all tiles, 1 the boundary tiles
// [0, n_boundary_tiles), 2 the others; op->range_begin >= 0 overrides it with an explicit tile range.
template <int N, class Params>
static void fill_common_params(Params &prm, bp5_operator_t op, double *dst, const double *src, double *dot_partials,
                               int which) {
  prm.cell_base = op->cell_base; prm.l2g_irr = op->l2g_irr;
  prm.src = src; prm.dst = dst;
  prm.tile_begin = which == 2 ? op->n_boundary_tiles : 0;
  prm.n_tiles = which == 1 ? op->n_boundary_tiles : op->n_tiles;      // end of the range
  if (op->range_begin >= 0) { prm.tile_begin = op->range_begin; prm.n_tiles = op->range_end; }
  prm.sy = op->od[0]; prm.sz = op->od[0] * op->od[1];
  prm.skip = op->skip_flag;
  prm.dot_partials = dot_partials;
  for (int q = 0; q < N; ++q) prm.wq[q] = op->tab.wq[q];
  fill_kernel_tables<N>(prm.tab, op->tab.B, op->tab.Dt);
}

// One launch of `kernel` over prm's tile range as a persistent grid: as many CTAs as fit on the device at once, at
// most one per tile and at most op->grid_cap; op->apply_grid receives the grid size (= number of fused-dot partials).
// carveout: the kernel's preferred shared-memory carve-out, cudaSharedmemCarveoutDefault to leave it alone.
template <auto kernel, class Params>
static int launch_cell_kernel(bp5_operator_t op, const Params &prm, int nt, size_t smem_bytes, int carveout) {
  // per instantiation and per device: function attributes belong to the device's context, and the C ABI allows
  // contexts on several devices in one process
  static int blocks_per_sm_of[64] = {0};
  int &blocks_per_sm = blocks_per_sm_of[op->ctx->device & 63];
  if (blocks_per_sm == 0) {
    BP5_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    if (carveout != cudaSharedmemCarveoutDefault)
      BP5_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carveout));
    int nb = 0;
    BP5_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, nt, smem_bytes));
    BP5_REQUIRE(nb > 0, "cell kernel does not fit on an SM");
    blocks_per_sm = nb;
  }
  if (prm.n_tiles <= prm.tile_begin) { op->apply_grid = 0; return BP5_OK; }
  long long grid = (long long)blocks_per_sm * op->ctx->sm_count;
  if (grid > prm.n_tiles - prm.tile_begin) grid = prm.n_tiles - prm.tile_begin;
  if (grid < 1) grid = 1;
  if (op->grid_cap > 0 && grid > op->grid_cap) grid = op->grid_cap;
  BP5_REQUIRE(grid <= kApplyPartialCap, "apply grid exceeds the partial-sum buffer");
  op->apply_grid = (int)grid;
  cudaStream_t stream = op->ctx->stream;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (op->profile) {
    if (op->prof_used + 2 > op->prof_events.size()) {
      for (int i = 0; i < 64; ++i) { cudaEvent_t e; BP5_CUDA(cudaEventCreate(&e)); op->prof_events.push_back(e); }
    }
    e0 = op->prof_events[op->prof_used++]; e1 = op->prof_events[op->prof_used++];
    BP5_CUDA(cudaEventRecord(e0, stream));
  }
  kernel<<<(unsigned)grid, nt, smem_bytes, stream>>>(prm);
  BP5_CHECK_LAUNCH();
  if (e1) BP5_CUDA(cudaEventRecord(e1, stream));
  op->ctx->launches++;
  return BP5_OK;
}

// One instantiation of the stored-metric kernel family (apply.cuh).  AFFINE: the constant-Jacobian kernel of an
// undeformed mesh with geometry on the fly; HANG: the kernels of a locally refined mesh; BLK: the merged CG's blocked
// layout (op->blk, set up by operator_setup_blocked).
template <int P, int QUAD, int HELM, int OWMODE, bool AFFINE = false, int HANG = 0, bool BLK = false>
static int launch(bp5_operator_t op, double *dst, const double *src, double *dot_partials, int which) {
  constexpr int CPT = TileCells<P>::value;
  using Cfg = ApplyCfg<P, CPT, 6 + HELM, AFFINE>;
  constexpr int N = P + 1;
  static_assert(HANG == 0 || !AFFINE, "hanging-node kernels stage the metric through shared memory");
  constexpr auto kernel = [] {
    if constexpr (HANG == 1) return bp5_apply_hang_kernel<P, QUAD, HELM, CPT, OWMODE>;
    else if constexpr (HANG == 2) return bp5_apply_strided_kernel<P, QUAD, HELM, CPT, OWMODE>;
    else return bp5_apply_kernel<P, QUAD, HELM, CPT, OWMODE, AFFINE, BLK>;
  }();
  ApplyParams<N> prm;
  fill_common_params<N>(prm, op, dst, src, dot_partials, which);
  prm.metric = op->metric;
  double hc[3];
  for (int d = 0; d < 3; ++d) hc[d] = (op->prob.upper[d] - op->prob.lower[d]) / op->prob.cells[d];
  prm.aff[0] = hc[1] * hc[2] / hc[0]; prm.aff[1] = hc[0] * hc[2] / hc[1]; prm.aff[2] = hc[0] * hc[1] / hc[2];
  prm.cell_mask = op->cell_mask;
  for (int cl = 0; cl < 8; ++cl) { prm.hang_sy[cl] = op->hang_sy[cl]; prm.hang_sz[cl] = op->hang_sz[cl]; }
  for (int sI = 0; sI < 2; ++sI)
    for (int i = 0; i < N * N; ++i) prm.hang[sI][i] = op->hanging_interp[sI][i];
  prm.blk_desc = op->blk_desc;
  prm.blk_stride = (int)(op->n_tiles * op->cells_per_tile);
  prm.blk_up_b = op->blk.ki * op->blk.nx; prm.blk_up_c = op->blk.ki * op->blk.ji;
  prm.blk_ji = op->blk.ji; prm.blk_plane = op->blk.nx * op->blk.ny;
  if constexpr (BLK) prm.cell_base = op->blk_desc;
  // all of the L1/shared array as shared memory (the kernel's working set is its tiles; the gathers are
  // served by L2): with the default carve-out the p=6 kernel gets 2 instead of 3 CTAs per SM.
  return launch_cell_kernel<kernel>(op, prm, Cfg::NT, Cfg::SMEM_BYTES, cudaSharedmemCarveoutMaxShared);
}

// Resident CTAs per SM and local-memory bytes (spills, stack) of the in-loop kernel of the merged CG (OVERWRITE = 2), in
// the lexicographic (BLK = false) or the blocked layout, with the launch attributes `launch` sets.
template <int P, int QUAD, int HELM, bool AFFINE, bool BLK>
static int cg_kernel_resources(int *ctas, size_t *local) {
  constexpr int CPT = TileCells<P>::value;
  using Cfg = ApplyCfg<P, CPT, 6 + HELM, AFFINE>;
  constexpr auto kernel = bp5_apply_kernel<P, QUAD, HELM, CPT, 2, AFFINE, BLK>;
  BP5_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_BYTES));
  BP5_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  BP5_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas, kernel, Cfg::NT, Cfg::SMEM_BYTES));
  cudaFuncAttributes fa;
  BP5_CUDA(cudaFuncGetAttributes(&fa, kernel));
  *local = fa.localSizeBytes;
  return BP5_OK;
}

// the same for op's kernel family (stored metric or affine) and degree, quadrature and operator
template <bool BLK>
static int op_cg_kernel_resources(bp5_operator_t op, int *ctas, size_t *local) {
  if (op->cell_kernel == CellKernel::kAffine)
    return with_degree(op->p, [&](auto P) {
      return with_value<0, 1>(op->prob.quadrature == BP5_QUAD_GLL,
                              [&](auto quad) { return cg_kernel_resources<P, quad, 0, true, BLK>(ctas, local); });
    });
  return with_degree(op->p, [&](auto P) {
    return with_quad_op(op, [&](auto quad, auto helm) { return cg_kernel_resources<P, quad, helm, false, BLK>(ctas, local); });
  });
}

// defined in apply_colored.cu / apply_hang.cu
int launch_colored(bp5_operator_t op, double *dst, const double *src, int mode, double *dp, int which);
int launch_hanging(bp5_operator_t op, double *dst, const double *src, int mode, double *dp, int which);

}  // namespace bp5
