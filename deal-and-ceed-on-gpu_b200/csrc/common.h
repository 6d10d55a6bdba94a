// Internal types shared by the translation units of libbp5b200.so.
// Product code: sm_100a only, no CPU fallback.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/bp5_b200.h"

namespace bp5 {

constexpr int kMaxDegree = 8;
constexpr int kApplyPartialCap = 4096;      // per-CTA partial sums of the cell kernel's fused dot product
constexpr int kConstrainedPartials = 148 * 8;   // blocks (= partial sums) of the Dirichlet-copy correction
constexpr int kMaxN = kMaxDegree + 1;

// ---- error plumbing --------------------------------------------------------
void set_error(const char *fmt, ...);
const char *get_error();

#define BP5_CUDA(call)                                                                  \
  do {                                                                                  \
    cudaError_t err__ = (call);                                                         \
    if (err__ != cudaSuccess) {                                                         \
      ::bp5::set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__,             \
                       cudaGetErrorString(err__));                                      \
      return BP5_ERR_CUDA;                                                              \
    }                                                                                   \
  } while (0)

#define BP5_CHECK_LAUNCH()                                                              \
  do {                                                                                  \
    cudaError_t err__ = cudaGetLastError();                                             \
    if (err__ != cudaSuccess) {                                                         \
      ::bp5::set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__,         \
                       cudaGetErrorString(err__));                                      \
      return BP5_ERR_CUDA;                                                              \
    }                                                                                   \
  } while (0)

#define BP5_REQUIRE(cond, msg)                                                          \
  do {                                                                                  \
    if (!(cond)) {                                                                      \
      ::bp5::set_error("%s (%s:%d)", msg, __FILE__, __LINE__);                          \
      return BP5_ERR_INVALID;                                                           \
    }                                                                                   \
  } while (0)

// ---- 1D tables (host) ------------------------------------------------------
// n = p+1.  All matrices row-major [row*n + col].
struct Tables1D {
  int n;                       // POD: lives in __constant__ memory too
  double xi[kMaxN];           // FE_Q support points: Gauss-Lobatto on [0,1]
  double xq[kMaxN], wq[kMaxN]; // quadrature points / weights on [0,1]
  double B[kMaxN * kMaxN];     // B[q][i]  = phi_i(xq_q)       (identity for GLL quadrature)
  double Dg[kMaxN * kMaxN];    // Dg[q][i] = phi_i'(xq_q)
  double Dt[kMaxN * kMaxN];    // Dt[q][r] = l_r'(xq_q), l_r = Lagrange basis through the QUADRATURE points
};
void make_tables(int degree, int quadrature, Tables1D &t);
void gauss_rule01(int n, double *x, double *w);
void lobatto_rule01(int n, double *x, double *w);
void lagrange_eval(int n, const double *nodes, double x, double *val, double *der);
void parent_child_interp(const Tables1D &t, double (*out)[kMaxN * kMaxN]);   // [s][a*n + b] = l_b((s + xi_a) / 2)

// device scratch of one CG solve (cg.cu): [CgState | dots partials | cell-kernel p.v partials | Dirichlet correction
// partials | update-kernel r.r partials | residual history]
struct CgState;
struct CgBuffers {
  CgState *st;
  double *partials;    // [kCgBlocks][7]
  double *ph;          // [kApplyPartialCap + kConstrainedPartials]
  double *rr;          // [kUpdatePartialCap][2]
  double *hist;        // [hist_len] or nullptr
};

// The merged CG's blocked DoF layout on one conforming block (blocked.cuh): [interior blocks | skeleton].  Each cell's
// (p-1)^3 interior DoFs are one contiguous block, in the cell processing order; the skeleton (lattice points with a
// coordinate on a cell face) comes in three classes, each affine in a cell's local coordinates:
//   A  points on z-face planes, lexicographic (x, y, plane);
//   B  points on y-face planes and not on a z-face plane, (x, non-face z, plane);
//   C  points on x-face planes only, (non-face y, non-face z, plane) -- y fastest, so a cell's x-face is read in runs.
// Interior DoFs are touched by one cell only and share no 32-byte sector with the skeleton's atomics.
struct BlockedLayout {
  int p = 0, nc[3] = {0, 0, 0};   // degree, cells per direction
  int nx = 0, ny = 0;             // lattice points in x and y (p nc + 1)
  int ki = 0, ji = 0;             // non-face lattice planes in z and in y: nc (p - 1)
  long long sa = 0, sb = 0, sc = 0, n = 0;   // starts of the classes A, B, C (sa = number of interior DoFs); size
};

// The family of cell kernels an operator runs, chosen once by apply_choose
enum class CellKernel {
  kStored,             // stored metric (apply.cuh); coloured and hanging-node variants follow cell order and refinement
  kAffine,             // geometry on the fly on an undeformed mesh: one constant Jacobian (apply.cuh, AFFINE)
  kOnTheFly,           // geometry on the fly, collocation + Poisson, four fields at once (apply_otf.cuh)
  kOnTheFlyGeneral,    // geometry on the fly, every quadrature / operator (apply_otfg.cuh)
};

// ---- handles ---------------------------------------------------------------
}  // namespace bp5

struct bp5_context_s {
  int device = 0;
  cudaStream_t stream = nullptr;
  int sm_count = 0;
  int64_t launches = 0;
  double *scratch = nullptr;      // small device scratch for reductions
  double *scratch_host = nullptr; // pinned
};

struct bp5_vector_s {
  bp5_context_t ctx = nullptr;
  int64_t n_owned = 0, n_ghost = 0;
  double *d = nullptr;
  bp5_operator_t owner = nullptr;   // operator whose initialize_dof_vector made it (its "partitioner"), or null
};

struct bp5_operator_s {
  bp5_context_t ctx = nullptr;
  bp5_problem_t prob{};
  bp5::Tables1D tab;
  int p = 0, n = 0;
  // this block
  int lc[3] = {0, 0, 0};        // local cells per direction
  int c0[3] = {0, 0, 0};        // first global cell
  int ld[3] = {0, 0, 0};        // local dofs per direction (owned + lower ghost layer)
  int has_lo[3] = {0, 0, 0};    // a lower neighbour owns the lower face
  int has_hi[3] = {0, 0, 0};
  int od[3] = {0, 0, 0};        // owned dofs per direction
  int64_t n_owned = 0, n_ghost = 0, n_global = 0, n_cells = 0;
  int64_t ghost_offset[8] = {0}; // start of ghost group m (1..7) relative to n_owned
  int64_t ghost_size[8] = {0};
  int cells_per_tile = 1;
  int apply_grid = 0;           // CTAs of the last cell-kernel launch (= number of fused-dot partial sums)
  bp5::CellKernel cell_kernel = bp5::CellKernel::kStored;
  int64_t n_tiles = 0;
  int64_t n_boundary_cells = 0;  // cells touching a lower ghost layer; they occupy tiles [0, n_boundary_tiles)
  int64_t n_boundary_tiles = 0;
  int64_t color_tile_begin[9] = {0};  // cell_order = BP5_CELL_ORDER_COLORED: tiles [begin[c], begin[c+1]) hold colour c
  int64_t tile_doubles = 0;     // metric doubles per tile (padded to a multiple of 2)
  // device data
  int *cell_base = nullptr;     // [n_tiles*cpt] per-cell dof descriptor: >= 0 affine base (idx = base + i + j*od0 +
                                // k*od0*od1), < 0: -(slot+1) into l2g_irr, INT_MIN: padding cell
  int *l2g_irr = nullptr;       // [n_irregular][n^3] explicit local dof indices (cells touching lower ghost layers)
  int64_t n_irregular = 0;
  // deal.II-layout arrays for user-written cell functors (built on first request)
  unsigned int *mf_l2g = nullptr, *mf_constraint_mask = nullptr;
  double *mf_inv_jacobian = nullptr, *mf_jxw = nullptr, *mf_q_points = nullptr;
  int mf_padding = 0;
  // the same arrays per parity colour of the cells (use_coloring): colour = px + 2 py + 4 pz
  bool mf_colors_built = false;
  unsigned int *mfc_l2g[8] = {nullptr}, *mfc_constraint_mask[8] = {nullptr};
  double *mfc_inv_jacobian[8] = {nullptr}, *mfc_jxw[8] = {nullptr}, *mfc_q_points[8] = {nullptr};
  int64_t mfc_n_cells[8] = {0};
  double *coords = nullptr;     // BP5_GEOM_ON_THE_FLY: nodal coordinates [3][n_owned + n_ghost] instead of the metric
  double *metric = nullptr;     // [tile][cpt][planes][n^3]; planes: 6 (Poisson) or 7 (Helmholtz: + a*JxW)
  int metric_planes = 6;
  int *constrained = nullptr;   // local owned indices of Dirichlet dofs
  // locally refined mesh (refine_lo/refine_hi of the problem): generic functor path only, see operator_setup_hanging
  bool hanging = false;
  void *hanging_cells = nullptr;                  // device int4[n_cells]: (lattice index x, y, z, level) per cell
  double *hanging_interp_dev = nullptr;           // device copy of hanging_interp
  int64_t hanging_affine_cells = 0;               // cells of a refined mesh with an affine descriptor
  int hang_sy[8] = {0}, hang_sz[8] = {0};         // stride classes of the affine cells of a refined mesh (cell_mask bits 8..10)
  unsigned int *cell_mask = nullptr;              // [n_tiles * cells_per_tile] constraint mask per cell slot (tuned kernel)
  double hanging_interp[2][bp5::kMaxN * bp5::kMaxN] = {};   // [s][a * n + b] = l_b((s + xi_a) / 2): parent-to-child, 1D
  std::vector<double> hanging_coords;             // [n_owned][3] mapped support point of every DoF
  int64_t n_constrained = 0;
  bool do_zero_out = true;
  std::string kernel_name;
  // CG work vectors (allocated on first solve)
  bp5_vector_t g = nullptr, d = nullptr, h = nullptr;
  bp5_vector_t xh = nullptr, bh = nullptr;  // device staging of bp5_cg_solve_host
  double *cg_scalars = nullptr; // device
  size_t cg_scalars_bytes = 0;
  bp5_vector_t cg_x = nullptr, cg_diag = nullptr;   // stepwise CG: caller's solution / diagonal
  int cg_hist_len = 0;
  bp5::CgBuffers cg_buf{};      // stepwise CG: cg_scalars as laid out by cg_step_begin
  bool cg_ph_valid = false;     // stepwise CG: the cell kernel left d.h partials for the next dots step
  int cg_update_grid = 0;       // stepwise CG: blocks (= r.r partials) of the last update step
  // merged CG in the blocked layout (operator_setup_blocked, built by the first solve that takes it)
  bp5::BlockedLayout blk{};
  int *blk_desc = nullptr;        // [4][n_tiles * cells_per_tile] per-cell starts in class A, B, C and of the interior
                                  // block; class A: kNoCell for tile padding
  int *blk_constrained = nullptr; // the Dirichlet list in the blocked layout
  bp5_vector_t blk_x = nullptr, blk_diag = nullptr;   // the solution and the diagonal in the blocked layout
  int blk_fits = -1;              // the blocked in-loop kernel keeps the lexicographic one's CTAs/SM, no more spill
                                  // (1 / 0, -1: not yet asked)
  // live per-launch timing of the cell kernel (bench.py roofline): events around every launch
  bool profile = false;
  std::vector<cudaEvent_t> prof_events;   // start/stop pairs
  size_t prof_used = 0;
  void *peer = nullptr;          // peer-memory transport state (peer.cu), or null
  bool peer_connected = false;
  const int *skip_flag = nullptr; // device word: when non-zero the cell loop is a no-op (CG converged)
  // overrides of the next cell-kernel launch (peer-memory CG, coloured cell order)
  long long range_begin = -1, range_end = -1;   // tile range instead of `which`
  int grid_cap = 0;                             // upper bound of the cell kernel's grid (colour passes), 0 = none
};

namespace bp5 {
// setup.cu
int operator_generic_data_hanging(bp5_operator_t op);   // the same arrays for a locally refined mesh, on first use
int operator_setup_hanging(bp5_operator_t op);      // locally refined mesh: numbering + generic-path arrays
void operator_plan_tiles(bp5_operator_t op);       // fills n_boundary_cells, n_boundary_tiles, n_tiles
int operator_setup_device(bp5_operator_t op);
int operator_assemble_rhs(bp5_operator_t op, double *b_dev);
int operator_l2_norm_sqr(bp5_operator_t op, const double *u_dev, double *out);
int operator_generic_data(bp5_operator_t op);
int operator_generic_data_colored(bp5_operator_t op);
int operator_diagonal(bp5_operator_t op, double *diag_dev, bool invert);
bool operator_blocked_supported(bp5_operator_t op);         // the merged CG can run in the blocked layout
int operator_setup_blocked(bp5_operator_t op);            // op->blk, blk_desc, blk_constrained (first call only)
int operator_export_coefficients(bp5_operator_t op, double *host_out);
int operator_export_coords(bp5_operator_t op, double *host_out);
int operator_export_global_indices(bp5_operator_t op, int64_t *host_out);
// apply.cu
int apply_choose(bp5_operator_t op);                 // picks the kernel family, cells_per_tile, tile plan + kernel name
// which: 0 all tiles, 1 boundary tiles only, 2 the others
int apply_cell_loop(bp5_operator_t op, double *dst, const double *src, bool overwrite_interior,
                    double *dot_partials = nullptr, int which = 0);
// the on-the-fly-geometry kernels (apply_otf.cu, apply_otfg.cu)
int apply_cell_loop_otf(bp5_operator_t op, double *dst, const double *src, int mode, double *dot_partials, int which);
int apply_cell_loop_otfg(bp5_operator_t op, double *dst, const double *src, int mode, double *dot_partials, int which);
// the merged CG's cell loop in the blocked layout (apply_blocked.cu): overwrite interior, per-CTA partials of src.(A src)
int apply_cell_loop_blocked(bp5_operator_t op, double *dst, const double *src, double *dot_partials);
int apply_blocked_kernel_resources(bp5_operator_t op, int *ctas, size_t *local);
// resident CTAs per SM and local-memory bytes of the merged CG's in-loop cell kernel, lexicographic or blocked
int apply_cg_kernel_resources(bp5_operator_t op, bool blocked, int *ctas, size_t *local);
// list: the Dirichlet DoFs in the layout of dst and src (op->constrained or op->blk_constrained)
int apply_copy_constrained_dot(bp5_operator_t op, const int *list, double *dst, const double *src, double *partials);
int apply_zero_skeleton(bp5_operator_t op, double *dst);
int apply_copy_constrained(bp5_operator_t op, double *dst, const double *src);
// vector.cu
int vec_fill(bp5_context_t ctx, double *d, int64_t n, double v);
int vec_axpy(bp5_context_t ctx, double *y, double s, double a, const double *x, int64_t n, int mode);
int vec_dot(bp5_context_t ctx, const double *x, const double *y, int64_t n, double *out);
int vec_all_zero(bp5_context_t ctx, const double *x, int64_t n, int *out);
// to_blocked: dst[blocked(t)] = scale * src[t]; otherwise dst[t] = scale * src[blocked(t)] (t lexicographic)
int vec_blocked_permute(bp5_context_t ctx, const BlockedLayout &L, double *dst, const double *src, double scale,
                        bool to_blocked);
// halo.cu
int halo_info(bp5_operator_t op, int64_t *send_count, int64_t *send_offset, int64_t *recv_count, int64_t *recv_offset);
int halo_pack(bp5_operator_t op, const double *vec, double *sendbuf);
int halo_unpack_add(bp5_operator_t op, double *vec, const double *recvbuf);
// peer.cu
int peer_export(bp5_operator_t op, int rank, int world, bp5_peer_info_t *out);
int peer_connect(bp5_operator_t op, const bp5_peer_info_t *all, const int *upper_rank, const int *lower_rank);
void peer_destroy(bp5_operator_t op);
int peer_forward(bp5_operator_t op, const double *vec, bool wait = true);   // wait: also wait for the lower neighbours' data
int peer_wait_forward(bp5_operator_t op);
int peer_reverse(bp5_operator_t op, const double *vec);
int peer_wait_add(bp5_operator_t op, double *vec);
int peer_allreduce(bp5_operator_t op, const double *local_dev, double *out_dev, int n_vals, bool honour_skip,
                   void *cg_state = nullptr, double *history = nullptr);
int peer_allreduce_host(bp5_operator_t op, double *vals, int n);
int peer_vmult(bp5_operator_t op, bp5_vector_t dst, bp5_vector_t src);
int peer_world_size(bp5_operator_t op);
int peer_update_ghost_values(bp5_operator_t op, bp5_vector_t vec);
int peer_compress_add(bp5_operator_t op, bp5_vector_t vec);
double *peer_scratch(bp5_operator_t op);
int peer_check(bp5_operator_t op);
int cg_solve_peer(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diag, int control, double tol,
                  int max_its, int *last_step, double *last_value, double *history, int history_len);
// cg.cu
// creates the work vectors g, d, h on first use and grows the device scratch to hold a residual history of hist_len;
// cb (may be null) receives its layout
int cg_buffers(bp5_operator_t op, int hist_len, CgBuffers *cb);
// return code and error text of a CG that ended in CgState::state `state` (1 success, 2 no convergence, 3 d.Ad == 0)
// after `it` iterations at residual `res`
int cg_status(int state, int it, double res);
int cg_step_begin(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diag, int control, double tol,
                  int max_its, double res0, int history_len);
int cg_step_update(bp5_operator_t op, int iteration);
int cg_step_apply_local(bp5_operator_t op);
int cg_step_constrained(bp5_operator_t op);
int cg_step_local_dots(bp5_operator_t op, double *sums_dev);
int cg_step_scalars(bp5_operator_t op, const double *sums_dev);
int cg_step_poll(bp5_operator_t op, int *state, int *it, double *res);
int cg_step_finish(bp5_operator_t op, double *history);
int cg_solve(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diag, int variant, int control,
             double tol, int max_its, int *last_step, double *last_value, double *history, int history_len);
}  // namespace bp5
