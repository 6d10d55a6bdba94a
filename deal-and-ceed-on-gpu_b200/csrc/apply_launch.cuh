// Host-side launch of one instantiation of the cell kernel (persistent grid sizing, parameters, profiling events).
// Shared by the translation units that hold the instantiations -- apply.cu (the shipped modes), apply_colored.cu (plain
// adds for the coloured cell order), apply_hang.cu (hanging-node constraints) -- which are separate files only to
// compile in parallel.
#pragma once
#include <cstdlib>

#include "apply.cuh"
#include "tile_cells.h"

namespace bp5 {

template <int P, int QUAD, int HELM, int OVERWRITE, int MLOAD, int HANG = 0>
static int launch(bp5_operator_t op, double *dst, const double *src, double *dot_partials, int which) {
  constexpr int CPT = TileCells<P>::value;
  using Cfg = ApplyCfg<P, CPT, 6 + HELM, MLOAD>;
  constexpr int N = P + 1;
  static_assert(HANG == 0 || MLOAD == 0, "hanging-node kernels stage the metric through shared memory");
  auto kernel = [] {
    if constexpr (HANG == 1) return bp5_apply_hang_kernel<P, QUAD, HELM, CPT, OVERWRITE>;
    else if constexpr (HANG == 2) return bp5_apply_strided_kernel<P, QUAD, HELM, CPT, OVERWRITE>;
    else return bp5_apply_kernel<P, QUAD, HELM, CPT, OVERWRITE, MLOAD>;
  }();
  // per instantiation and per device: function attributes belong to the device's context, and the C ABI allows
  // contexts on several devices in one process
  static int blocks_per_sm_of[64] = {0};
  int &blocks_per_sm = blocks_per_sm_of[op->ctx->device & 63];
  if (blocks_per_sm == 0) {
    BP5_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_BYTES));
    // all of the L1/shared array as shared memory (the kernel's working set is its tiles; the gathers are
    // served by L2): with the default carve-out the p=6 kernel gets 2 instead of 3 CTAs per SM.
    // BP5_CARVEOUT=<percent> overrides for tuning runs.
    int carve = cudaSharedmemCarveoutMaxShared;
    if (const char *cv = getenv("BP5_CARVEOUT")) carve = atoi(cv);
    BP5_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carve));
    int nb = 0;
    BP5_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, Cfg::NT, Cfg::SMEM_BYTES));
    BP5_REQUIRE(nb > 0, "apply kernel does not fit on an SM");
    blocks_per_sm = nb;
  }
  ApplyParams<N> prm;
  prm.metric = op->metric; prm.cell_base = op->cell_base; prm.l2g_irr = op->l2g_irr;
  prm.src = src; prm.dst = dst;
  prm.tile_begin = which == 2 ? op->n_boundary_tiles : 0;
  prm.n_tiles = which == 1 ? op->n_boundary_tiles : op->n_tiles;      // end of the range
  if (op->range_begin >= 0) { prm.tile_begin = op->range_begin; prm.n_tiles = op->range_end; }   // explicit tile range
  cudaStream_t stream = op->ctx->stream;
  prm.sy = op->od[0]; prm.sz = op->od[0] * op->od[1];
  if (prm.n_tiles <= prm.tile_begin) { op->apply_grid = 0; return BP5_OK; }
  prm.skip = op->skip_flag;
  prm.dot_partials = dot_partials;
  {
    double hc[3];
    for (int d = 0; d < 3; ++d) hc[d] = (op->prob.upper[d] - op->prob.lower[d]) / op->prob.cells[d];
    prm.aff[0] = hc[1] * hc[2] / hc[0]; prm.aff[1] = hc[0] * hc[2] / hc[1]; prm.aff[2] = hc[0] * hc[1] / hc[2];
    for (int q = 0; q < N; ++q) prm.wq[q] = op->tab.wq[q];
  }
  prm.cell_mask = op->cell_mask;
  for (int cl = 0; cl < 8; ++cl) { prm.hang_sy[cl] = op->hang_sy[cl]; prm.hang_sz[cl] = op->hang_sz[cl]; }
  for (int sI = 0; sI < 2; ++sI)
    for (int i = 0; i < N * N; ++i) prm.hang[sI][i] = op->hanging_interp[sI][i];
  fill_kernel_tables<N>(prm.tab, op->tab.B, op->tab.Dt);
  long long grid = (long long)blocks_per_sm * op->ctx->sm_count;
  if (grid > prm.n_tiles - prm.tile_begin) grid = prm.n_tiles - prm.tile_begin;
  if (grid < 1) grid = 1;
  if (op->grid_cap > 0 && grid > op->grid_cap) grid = op->grid_cap;
  BP5_REQUIRE(grid <= kApplyPartialCap, "apply grid exceeds the partial-sum buffer");
  op->apply_grid = (int)grid;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (op->profile) {
    if (op->prof_used + 2 > op->prof_events.size()) {
      for (int i = 0; i < 64; ++i) { cudaEvent_t e; BP5_CUDA(cudaEventCreate(&e)); op->prof_events.push_back(e); }
    }
    e0 = op->prof_events[op->prof_used++]; e1 = op->prof_events[op->prof_used++];
    BP5_CUDA(cudaEventRecord(e0, stream));
  }
  kernel<<<(unsigned)grid, Cfg::NT, Cfg::SMEM_BYTES, stream>>>(prm);
  BP5_CHECK_LAUNCH();
  if (e1) BP5_CUDA(cudaEventRecord(e1, stream));
  op->ctx->launches++;
  return BP5_OK;
}


// the dispatch over quadrature and operator for one degree / one OWMODE / one HANG value
#define BP5_LAUNCH_QH(P, M, MLOAD, HANG)                                                                              \
  (gll ? (helm ? launch<P, 1, 1, M, MLOAD, HANG>(op, dst, src, dp, which) : launch<P, 1, 0, M, MLOAD, HANG>(op, dst, src, dp, which)) \
       : (helm ? launch<P, 0, 1, M, MLOAD, HANG>(op, dst, src, dp, which) : launch<P, 0, 0, M, MLOAD, HANG>(op, dst, src, dp, which)))

// defined in apply_colored.cu / apply_hang.cu
int launch_colored(bp5_operator_t op, double *dst, const double *src, int mode, double *dp, int which);
int launch_hanging(bp5_operator_t op, double *dst, const double *src, int mode, double *dp, int which);

}  // namespace bp5
