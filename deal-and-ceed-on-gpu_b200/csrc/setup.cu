// Device-side setup of one mesh block: what the reference obtains from
// CUDAWrappers::MatrixFree::reinit (bp5/step-64.cu:248) [UPSTREAM] and
// evaluate_coefficients(JacobianFunctor) (bp5/step-64.cu:84-114, 256-258):
//   local_to_global map, Jacobians of the MappingQGeneric(p) geometry at the
//   quadrature points, the merged symmetric coefficient G = JxW J^-1 J^-T
//   (planes xx,yy,zz,xy,xz,yz), the Dirichlet set, and the right-hand side of
//   assemble_rhs (bp5/step-64.cu:372-418).
// Everything is generated on the GPU from the analytic mesh description; no
// O(n_dofs) host arrays are built except the Dirichlet index list.
#include <algorithm>
#include <climits>
#include <cmath>
#include <vector>

#include "blocked.cuh"

namespace bp5 {

struct BlockGeom {
  int n, p;
  int lc[3], c0[3], gc[3];      // local cells, first global cell, global cells
  int ld[3], hlo[3], od[3];     // local dofs/dir, lower-ghost flags, owned dofs/dir
  long long n_owned;
  long long goff[8];            // ghost group offsets (relative to n_owned)
  double lo[3], L[3], h[3];     // domain corner, extent, cell size
  int deform; double eps;
  int planes;                   // 6 (Poisson) or 7 (Helmholtz)
  int cpt; long long tile_doubles; // metric layout [tile][cpt][planes][n3], tile stride padded to 16 B
};

__constant__ Tables1D c_tab;

__device__ __forceinline__ long long local_dof_index(const BlockGeom &g, int i, int j, int k) {
  const int bx = i < g.hlo[0], by = j < g.hlo[1], bz = k < g.hlo[2];
  if (!(bx | by | bz))
    return (i - g.hlo[0]) + (long long)g.od[0] * ((j - g.hlo[1]) + (long long)g.od[1] * (k - g.hlo[2]));
  const int m = bx | (by << 1) | (bz << 2);
  const int e0 = bx ? 1 : g.od[0], e1 = by ? 1 : g.od[1];
  const int q0 = bx ? 0 : i - g.hlo[0], q1 = by ? 0 : j - g.hlo[1], q2 = bz ? 0 : k - g.hlo[2];
  return g.n_owned + g.goff[m] + q0 + (long long)e0 * (q1 + (long long)e1 * q2);
}

__device__ __forceinline__ void map_point(const BlockGeom &g, const double *x, double *y) {
  if (g.deform == 0) { y[0] = x[0]; y[1] = x[1]; y[2] = x[2]; return; }
  double s = 1.0;
  for (int d = 0; d < 3; ++d) s *= sin(M_PI * (x[d] - g.lo[d]) / g.L[d]);
  for (int d = 0; d < 3; ++d) y[d] = x[d] + g.eps * g.L[d] * s;
}

// Jacobian of the degree-p mapping at the n^3 points of a 1D rule given by the
// matrices Bm (values) / Dm (derivatives) [q][i]: three sum-factorised passes
// per coordinate.  One thread per point.  smem: X[3][n3] + 5 work arrays.
// On return J[d][e] and xr[d] hold this thread's point.
__device__ void cell_jacobian(const BlockGeom &g, const double *Bm, const double *Dm, double *sm, int cx, int cy,
                              int cz, double J[3][3], double xr[3]) {
  const int n = g.n, n2 = n * n, n3 = n2 * n;
  const int t = threadIdx.x;
  const int i = t % n, j = (t / n) % n, k = t / n2;
  double *X = sm, *tD = sm + 3 * n3, *tB = tD + n3, *tDB = tB + n3, *tBD = tDB + n3, *tBB = tBD + n3;
  if (t < n3) {
    const int c[3] = {cx, cy, cz};
    const int loc[3] = {i, j, k};
    double x[3], y[3];
    for (int d = 0; d < 3; ++d) x[d] = g.lo[d] + g.h[d] * (c[d] + c_tab.xi[loc[d]]);
    map_point(g, x, y);
    for (int d = 0; d < 3; ++d) X[d * n3 + t] = y[d];
  }
  __syncthreads();
  for (int d = 0; d < 3; ++d) {
    if (t < n3) {
      double sD = 0.0, sB = 0.0;
      for (int m = 0; m < n; ++m) {
        const double v = X[d * n3 + (k * n + j) * n + m];
        sD += Dm[i * n + m] * v; sB += Bm[i * n + m] * v;
      }
      tD[t] = sD; tB[t] = sB;
    }
    __syncthreads();
    if (t < n3) {
      double sDB = 0.0, sBD = 0.0, sBB = 0.0;
      for (int m = 0; m < n; ++m) {
        const double vD = tD[(k * n + m) * n + i], vB = tB[(k * n + m) * n + i];
        sDB += Bm[j * n + m] * vD; sBD += Dm[j * n + m] * vB; sBB += Bm[j * n + m] * vB;
      }
      tDB[t] = sDB; tBD[t] = sBD; tBB[t] = sBB;
    }
    __syncthreads();
    if (t < n3) {
      double j0 = 0.0, j1 = 0.0, j2 = 0.0, xv = 0.0;
      for (int m = 0; m < n; ++m) {
        const int a = (m * n + j) * n + i;
        j0 += Bm[k * n + m] * tDB[a]; j1 += Bm[k * n + m] * tBD[a];
        j2 += Dm[k * n + m] * tBB[a]; xv += Bm[k * n + m] * tBB[a];
      }
      J[d][0] = j0; J[d][1] = j1; J[d][2] = j2; xr[d] = xv;
    }
    __syncthreads();
  }
}

__device__ __forceinline__ double det3(const double J[3][3]) {
  return J[0][0] * (J[1][1] * J[2][2] - J[1][2] * J[2][1]) - J[0][1] * (J[1][0] * J[2][2] - J[1][2] * J[2][0]) +
         J[0][2] * (J[1][0] * J[2][1] - J[1][1] * J[2][0]);
}

// The merged coefficient G = JxW J^-1 J^-T (+ a(x) JxW for Helmholtz) of lattice cell (cx, cy, cz) of `g` at this
// thread's quadrature point, written at processing-order position `slot` of the metric tiles (whole CTA:
// cell_jacobian synchronises).
__device__ void write_cell_metric(const BlockGeom &g, double *sm, int cx, int cy, int cz, long long slot,
                                  double *__restrict__ metric) {
  const int n = g.n, n2 = n * n, n3 = n2 * n;
  const int t = threadIdx.x;
  const int i = t % n, j = (t / n) % n, k = t / n2;
  double J[3][3], xr[3];
  cell_jacobian(g, c_tab.B, c_tab.Dg, sm, cx, cy, cz, J, xr);
  if (t >= n3) return;
  const double det = det3(J);
  const double id = 1.0 / det;
  double I[3][3];   // I[d][f] = d xi_d / d x_f
  I[0][0] = (J[1][1] * J[2][2] - J[1][2] * J[2][1]) * id;
  I[0][1] = (J[0][2] * J[2][1] - J[0][1] * J[2][2]) * id;
  I[0][2] = (J[0][1] * J[1][2] - J[0][2] * J[1][1]) * id;
  I[1][0] = (J[1][2] * J[2][0] - J[1][0] * J[2][2]) * id;
  I[1][1] = (J[0][0] * J[2][2] - J[0][2] * J[2][0]) * id;
  I[1][2] = (J[0][2] * J[1][0] - J[0][0] * J[1][2]) * id;
  I[2][0] = (J[1][0] * J[2][1] - J[1][1] * J[2][0]) * id;
  I[2][1] = (J[0][1] * J[2][0] - J[0][0] * J[2][1]) * id;
  I[2][2] = (J[0][0] * J[1][1] - J[0][1] * J[1][0]) * id;
  const double jxw = det * c_tab.wq[i] * c_tab.wq[j] * c_tab.wq[k];
  // JacobianFunctor, bp5/step-64.cu:98-113
  double G[6];
  int pl = 3;
  for (int d = 0; d < 3; ++d) {
    G[d] = jxw * (I[d][0] * I[d][0] + I[d][1] * I[d][1] + I[d][2] * I[d][2]);
    for (int e = d + 1; e < 3; ++e, ++pl) G[pl] = jxw * (I[d][0] * I[e][0] + I[d][1] * I[e][1] + I[d][2] * I[e][2]);
  }
  double *out = metric + (slot / g.cpt) * g.tile_doubles + (slot % g.cpt) * (long long)g.planes * n3 + t;
  for (int c = 0; c < 6; ++c) out[(long long)c * n3] = G[c];
  if (g.planes == 7) {
    // VaryingCoefficientFunctor (step-64/step-64.cu:100-118) times JxW (submit_value,
    // bp5/fe_evaluation_gl.h:297-300)
    const double p2 = xr[0] * xr[0] + xr[1] * xr[1] + xr[2] * xr[2];
    out[6LL * n3] = 10.0 / (0.05 + 2.0 * p2) * jxw;
  }
}

// One block per local cell (lexicographic); `slot` is the cell's position in the processing order
// (cell_slot()).  Writes metric[tile][cell in tile][planes][n3] at that position and, for
// irregular cells (cell_base < 0), the explicit index table l2g_irr[table][n3].
__global__ void setup_cells_kernel(BlockGeom g, const int *__restrict__ cell_base, const long long *__restrict__ slot_of,
                                   int *__restrict__ l2g_irr, double *__restrict__ metric) {
  extern __shared__ double sm[];
  const int n = g.n, n2 = n * n, n3 = n2 * n;
  const long long cell = blockIdx.x;
  const int lcx = cell % g.lc[0], lcy = (cell / g.lc[0]) % g.lc[1], lcz = cell / ((long long)g.lc[0] * g.lc[1]);
  const int t = threadIdx.x;
  const int i = t % n, j = (t / n) % n, k = t / n2;
  const long long slot = slot_of[cell];
  const int base = cell_base[slot];
  if (t < n3 && base < 0)
    l2g_irr[(long long)(-(base + 1)) * n3 + t] =
        (int)local_dof_index(g, lcx * g.p + i, lcy * g.p + j, lcz * g.p + k);
  if (metric == nullptr) return;     // geometry on the fly: only the index tables are needed (uniform per block)
  write_cell_metric(g, sm, g.c0[0] + lcx, g.c0[1] + lcy, g.c0[2] + lcz, slot, metric);
}

// Right-hand side b_i = int phi_i * 1 with QGauss(p+1) (c_tab must hold the
// GAUSS tables).  Loops over the local cells plus one halo layer of cells above
// each upper face that has a neighbour, and adds only into OWNED dofs, so no
// ghost exchange is needed.  Dirichlet rows stay zero.
__global__ void rhs_kernel(BlockGeom g, int ex, int ey, int ez, double *__restrict__ b) {
  extern __shared__ double sm[];
  const int n = g.n, n2 = n * n, n3 = n2 * n;
  const long long cell = blockIdx.x;
  const int lcx = cell % ex, lcy = (cell / ex) % ey, lcz = cell / ((long long)ex * ey);
  const int t = threadIdx.x;
  const int i = t % n, j = (t / n) % n, k = t / n2;
  double J[3][3], xr[3];
  cell_jacobian(g, c_tab.B, c_tab.Dg, sm, g.c0[0] + lcx, g.c0[1] + lcy, g.c0[2] + lcz, J, xr);
  double *w0 = sm, *w1 = sm + n3;
  if (t < n3) w0[t] = det3(J) * c_tab.wq[i] * c_tab.wq[j] * c_tab.wq[k];
  __syncthreads();
  // v_i = sum_q B[q][i] w_q, three transposed passes
  if (t < n3) { double s = 0; for (int m = 0; m < n; ++m) s += c_tab.B[m * n + i] * w0[(k * n + j) * n + m]; w1[t] = s; }
  __syncthreads();
  if (t < n3) { double s = 0; for (int m = 0; m < n; ++m) s += c_tab.B[m * n + j] * w1[(k * n + m) * n + i]; w0[t] = s; }
  __syncthreads();
  if (t < n3) {
    double s = 0; for (int m = 0; m < n; ++m) s += c_tab.B[m * n + k] * w0[(m * n + j) * n + i];
    const int li = lcx * g.p + i, lj = lcy * g.p + j, lk = lcz * g.p + k;   // local dof coords (may exceed ld)
    const int gi = g.c0[0] * g.p + li, gj = g.c0[1] * g.p + lj, gk = g.c0[2] * g.p + lk;
    const bool owned = li >= g.hlo[0] && lj >= g.hlo[1] && lk >= g.hlo[2] && li < g.ld[0] && lj < g.ld[1] && lk < g.ld[2];
    const bool bdry = gi == 0 || gj == 0 || gk == 0 || gi == g.gc[0] * g.p || gj == g.gc[1] * g.p || gk == g.gc[2] * g.p;
    if (owned && !bdry) atomicAdd(&b[local_dof_index(g, li, lj, lk)], s);
  }
}

// coordinates + global lexicographic index of every local dof (owned, then ghost); soa: coordinate planes
// x[], y[], z[] of n_local entries each (what the on-the-fly kernel gathers) instead of xyz triples
__global__ void dof_info_kernel(BlockGeom g, double *__restrict__ xyz, long long *__restrict__ gidx, long long soa = 0) {
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long tot = (long long)g.ld[0] * g.ld[1] * g.ld[2];
  if (t >= tot) return;
  const int i = t % g.ld[0], j = (t / g.ld[0]) % g.ld[1], k = t / ((long long)g.ld[0] * g.ld[1]);
  const long long li = local_dof_index(g, i, j, k);
  const int loc[3] = {i, j, k};
  double x[3], y[3];
  long long gl[3];
  for (int d = 0; d < 3; ++d) {
    int c = loc[d] / g.p, l = loc[d] % g.p;
    if (c == g.lc[d]) { c -= 1; l = g.p; }
    x[d] = g.lo[d] + g.h[d] * (g.c0[d] + c + c_tab.xi[l]);
    gl[d] = (long long)g.c0[d] * g.p + loc[d];
  }
  map_point(g, x, y);
  if (xyz && soa) { xyz[li] = y[0]; xyz[soa + li] = y[1]; xyz[2 * soa + li] = y[2]; }
  else if (xyz) { xyz[3 * li] = y[0]; xyz[3 * li + 1] = y[1]; xyz[3 * li + 2] = y[2]; }
  if (gidx) gidx[li] = gl[0] + ((long long)g.gc[0] * g.p + 1) * (gl[1] + ((long long)g.gc[1] * g.p + 1) * gl[2]);
}

static BlockGeom make_geom(bp5_operator_t op) {
  BlockGeom g{};
  g.n = op->n; g.p = op->p;
  for (int d = 0; d < 3; ++d) {
    g.lc[d] = op->lc[d]; g.c0[d] = op->c0[d]; g.gc[d] = op->prob.cells[d];
    g.ld[d] = op->ld[d]; g.hlo[d] = op->has_lo[d]; g.od[d] = op->od[d];
    g.lo[d] = op->prob.lower[d]; g.L[d] = op->prob.upper[d] - op->prob.lower[d];
    g.h[d] = g.L[d] / op->prob.cells[d];
  }
  g.n_owned = op->n_owned;
  for (int m = 0; m < 8; ++m) g.goff[m] = op->ghost_offset[m];
  g.deform = op->prob.deformation; g.eps = op->prob.deformation_eps;
  g.planes = op->metric_planes;
  g.cpt = op->cells_per_tile;
  g.tile_doubles = op->tile_doubles;
  return g;
}

// Processing order of the cells (= order of cell_base and of the metric tiles): the cells that touch a
// lower ghost layer ("boundary" cells: the only ones that read ghost values of src and write ghost
// entries of dst) come first, padded to whole tiles, then all others in lexicographic order.  The cell
// loop can then run [0, n_boundary_tiles) between the two halves of the halo exchange and
// [n_boundary_tiles, n_tiles) concurrently with it (MatrixFree's overlap_communication_computation,
// bp5/step-64.cu:241).  On a single block there are no boundary cells and the order is lexicographic.
static bool cell_is_boundary(const bp5_operator_t op, int cx, int cy, int cz) {
  return (cx == 0 && op->has_lo[0]) || (cy == 0 && op->has_lo[1]) || (cz == 0 && op->has_lo[2]);
}

// Colour of a cell in the deterministic mode (cell_order = BP5_CELL_ORDER_COLORED): the parity of its three
// indices.  Cells of one colour share no DoF (neighbours differ by one in at least one index), so a pass over one
// colour can add into dst with plain read-modify-writes; the eight passes run one after the other.  This is
// MatrixFree::AdditionalData::use_coloring (bp5/step-64.cu:243 sets it to false and takes the atomics).
static int cell_color(int cx, int cy, int cz) { return (cx & 1) | ((cy & 1) << 1) | ((cz & 1) << 2); }

void operator_plan_tiles(bp5_operator_t op) {
  const int cpt = op->cells_per_tile;
  if (op->hanging) {
    // locally refined mesh (one block): the cells that need the constraint exchange or an index table
    // (n_boundary_cells, counted by operator_setup_hanging) first, padded to whole tiles, then the affine ones
    op->n_boundary_tiles = (op->n_boundary_cells + cpt - 1) / cpt;
    op->n_tiles = op->n_boundary_tiles + (op->n_cells - op->n_boundary_cells + cpt - 1) / cpt;
    return;
  }
  if (op->prob.cell_order == BP5_CELL_ORDER_COLORED) {
    // colour-major order, every colour padded to whole tiles (single block: no boundary cells)
    op->n_boundary_cells = 0;
    op->n_boundary_tiles = 0;
    op->color_tile_begin[0] = 0;
    for (int c = 0; c < 8; ++c) {
      int64_t cnt = 1;
      for (int d = 0; d < 3; ++d) cnt *= ((c >> d) & 1) ? op->lc[d] / 2 : (op->lc[d] + 1) / 2;
      op->color_tile_begin[c + 1] = op->color_tile_begin[c] + (cnt + cpt - 1) / cpt;
    }
    op->n_tiles = op->color_tile_begin[8];
    return;
  }
  // boundary cells: all cells minus those whose three indices are >= has_lo
  int64_t inner = 1;
  for (int d = 0; d < 3; ++d) inner *= op->lc[d] - op->has_lo[d];
  const int64_t n_b = op->n_cells - inner;
  op->n_boundary_cells = n_b;
  op->n_boundary_tiles = (n_b + cpt - 1) / cpt;
  op->n_tiles = op->n_boundary_tiles + (inner + cpt - 1) / cpt;
}

// Slot (position in the processing order) of every local cell, cells numbered lexicographically.
static void cell_slots(const bp5_operator_t op, std::vector<long long> &slot_of) {
  slot_of.resize((size_t)op->n_cells);
  const bool colored = op->prob.cell_order == BP5_CELL_ORDER_COLORED;
  int64_t next_c[8];
  for (int c = 0; c < 8; ++c) next_c[c] = colored ? op->color_tile_begin[c] * op->cells_per_tile : 0;
  int64_t cell = 0, next_b = 0, next_i = op->n_boundary_tiles * op->cells_per_tile;
  for (int cz = 0; cz < op->lc[2]; ++cz)
    for (int cy = 0; cy < op->lc[1]; ++cy)
      for (int cx = 0; cx < op->lc[0]; ++cx, ++cell)
        slot_of[cell] = colored ? next_c[cell_color(cx, cy, cz)]++ : cell_is_boundary(op, cx, cy, cz) ? next_b++ : next_i++;
}

int operator_setup_device(bp5_operator_t op) {
  bp5_context_t ctx = op->ctx;
  const int n = op->n, n3 = n * n * n;
  const BlockGeom g = make_geom(op);
  const int64_t padded_cells = op->n_tiles * op->cells_per_tile;
  // per-cell dof descriptors: affine base for regular cells, slot of an explicit
  // table for cells that touch a lower ghost layer, INT_MIN for tile padding
  std::vector<int> base((size_t)padded_cells, INT_MIN);
  std::vector<long long> slot_of;
  cell_slots(op, slot_of);
  int64_t n_irr = 0;
  {
    const int p = op->p;
    int64_t cell = 0;
    for (int cz = 0; cz < op->lc[2]; ++cz)
      for (int cy = 0; cy < op->lc[1]; ++cy)
        for (int cx = 0; cx < op->lc[0]; ++cx, ++cell) {
          const int64_t slot = slot_of[cell];
          if (cell_is_boundary(op, cx, cy, cz))
            base[slot] = -(int)(n_irr++) - 1;
          else
            base[slot] = (int)((cx * p - op->has_lo[0]) +
                               (int64_t)op->od[0] * ((cy * p - op->has_lo[1]) + (int64_t)op->od[1] * (cz * p - op->has_lo[2])));
        }
  }
  op->n_irregular = n_irr;
  BP5_CUDA(cudaMalloc(&op->cell_base, sizeof(int) * padded_cells));
  BP5_CUDA(cudaMemcpyAsync(op->cell_base, base.data(), sizeof(int) * padded_cells, cudaMemcpyHostToDevice, ctx->stream));
  long long *slot_dev = nullptr;
  BP5_CUDA(cudaMalloc(&slot_dev, sizeof(long long) * op->n_cells));
  BP5_CUDA(cudaMemcpyAsync(slot_dev, slot_of.data(), sizeof(long long) * op->n_cells, cudaMemcpyHostToDevice, ctx->stream));
  BP5_CUDA(cudaMalloc(&op->l2g_irr, sizeof(int) * std::max<int64_t>(n_irr, 1) * n3));
  const bool otf = op->prob.geometry_mode == BP5_GEOM_ON_THE_FLY;
  BP5_CUDA(cudaMemcpyToSymbolAsync(c_tab, &op->tab, sizeof(Tables1D), 0, cudaMemcpyHostToDevice, ctx->stream));
  if (!otf) {
    const size_t mbytes = sizeof(double) * op->n_tiles * op->tile_doubles;
    BP5_CUDA(cudaMalloc(&op->metric, mbytes));
    BP5_CUDA(cudaMemsetAsync(op->metric, 0, mbytes, ctx->stream));
  } else {
    // nodal coordinates of every local DoF (the mapped support points), three planes
    const long long n_local = op->n_owned + op->n_ghost;
    BP5_CUDA(cudaMalloc(&op->coords, sizeof(double) * 3 * n_local));
    const long long tot = (long long)op->ld[0] * op->ld[1] * op->ld[2];
    dof_info_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, ctx->stream>>>(g, op->coords, nullptr, n_local);
    BP5_CHECK_LAUNCH();
    ctx->launches++;
  }
  const int threads = ((n3 + 31) / 32) * 32;
  const size_t smem = sizeof(double) * 8 * n3;
  setup_cells_kernel<<<(unsigned)op->n_cells, threads, smem, ctx->stream>>>(g, op->cell_base, slot_dev, op->l2g_irr,
                                                                            op->metric);
  BP5_CHECK_LAUNCH();
  ctx->launches++;

  // Dirichlet set: owned dofs on the global boundary (boundary id 0 = whole
  // boundary, bp5/step-64.cu:354-357), ascending local index.
  std::vector<int> cons;
  const long long G[3] = {(long long)op->prob.cells[0] * op->p, (long long)op->prob.cells[1] * op->p,
                          (long long)op->prob.cells[2] * op->p};
  for (int k = op->has_lo[2]; k < op->ld[2]; ++k) {
    const long long gk = (long long)op->c0[2] * op->p + k;
    for (int j = op->has_lo[1]; j < op->ld[1]; ++j) {
      const long long gj = (long long)op->c0[1] * op->p + j;
      const bool plane_b = gk == 0 || gk == G[2] || gj == 0 || gj == G[1];
      const long long row = (long long)op->od[0] * ((j - op->has_lo[1]) + (long long)op->od[1] * (k - op->has_lo[2]));
      if (plane_b) {
        for (int i = op->has_lo[0]; i < op->ld[0]; ++i) cons.push_back((int)(row + i - op->has_lo[0]));
      } else {
        if (op->c0[0] == 0 && !op->has_lo[0]) cons.push_back((int)row);
        if ((long long)op->c0[0] * op->p + op->ld[0] - 1 == G[0]) cons.push_back((int)(row + op->od[0] - 1));
      }
    }
  }
  op->n_constrained = (int64_t)cons.size();
  if (!cons.empty()) {
    BP5_CUDA(cudaMalloc(&op->constrained, sizeof(int) * cons.size()));
    BP5_CUDA(cudaMemcpyAsync(op->constrained, cons.data(), sizeof(int) * cons.size(), cudaMemcpyHostToDevice, ctx->stream));
  }
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  cudaFree(slot_dev);
  return BP5_OK;
}

// The merged CG takes the blocked layout on one conforming block in the default cell order, with a cell kernel of
// apply.cuh (stored metric, or the affine fast path of geometry on the fly), where the blocked in-loop kernel is
// resident with at least as many CTAs per SM as the lexicographic one and spills no more.  (Its index arithmetic costs
// registers: without that condition p = 3 and p = 7 with Gauss quadrature on the affine path would lose a CTA per SM,
// and p = 8 would spill.)
bool operator_blocked_supported(bp5_operator_t op) {
  if (op->n_ghost != 0 || op->hanging || op->peer || op->prob.cell_order != BP5_CELL_ORDER_DEFAULT) return false;
  if (op->cell_kernel != CellKernel::kStored && op->cell_kernel != CellKernel::kAffine) return false;
  for (int d = 0; d < 3; ++d)
    if (op->lc[d] != op->prob.cells[d] || op->has_lo[d] || op->has_hi[d]) return false;
  // What the layout saves is DRAM traffic (the zero-fill and the L2 fill of interior h).  Where the iteration's working
  // set -- five vectors and the metric -- stays in L2 there is none, and the lexicographic path keeps the CG's sums in
  // the order of the library's other CG paths (the blocked order alone moves x by ~1e-8 after ~80 iterations).
  int l2 = 0;
  if (cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, op->ctx->device) != cudaSuccess) return false;
  const double working_set = 8.0 * (5.0 * op->n_owned + (op->metric ? (double)op->n_tiles * op->tile_doubles : 0.0));
  if (working_set <= l2) return false;
  if (op->blk_fits < 0) {
    int c_lex = 0, c_blk = 0;
    size_t l_lex = 0, l_blk = 0;
    if (apply_cg_kernel_resources(op, false, &c_lex, &l_lex) != BP5_OK ||
        apply_cg_kernel_resources(op, true, &c_blk, &l_blk) != BP5_OK)
      return false;   // the error is reported by the launch of the lexicographic kernel
    op->blk_fits = c_blk >= c_lex && l_blk <= l_lex;
  }
  return op->blk_fits == 1;
}

int operator_setup_blocked(bp5_operator_t op) {
  if (op->blk_desc) return BP5_OK;
  BP5_REQUIRE(operator_blocked_supported(op), "the blocked layout needs one conforming block in the default cell order");
  bp5_context_t ctx = op->ctx;
  const BlockedLayout L = make_blocked_layout(op->p, op->lc);
  BP5_REQUIRE(L.n == op->n_owned, "blocked layout does not cover the owned DoFs");
  const int p = op->p;
  // single block, default order: cell slot = lexicographic cell number
  const int64_t padded = op->n_tiles * op->cells_per_tile;
  std::vector<int> desc((size_t)(4 * padded), 0);
  for (int64_t s = op->n_cells; s < padded; ++s) desc[s] = INT_MIN;   // kNoCell
  int64_t cell = 0;
  for (int cz = 0; cz < op->lc[2]; ++cz)
    for (int cy = 0; cy < op->lc[1]; ++cy)
      for (int cx = 0; cx < op->lc[0]; ++cx, ++cell) {
        desc[cell] = (int)(L.sa + ((int64_t)cz * L.ny + (int64_t)cy * p) * L.nx + (int64_t)cx * p);
        desc[padded + cell] = (int)(L.sb + ((int64_t)cy * L.ki + (int64_t)cz * (p - 1)) * L.nx + (int64_t)cx * p);
        desc[2 * padded + cell] = (int)(L.sc + ((int64_t)cx * L.ki + (int64_t)cz * (p - 1)) * L.ji + (int64_t)cy * (p - 1));
        desc[3 * padded + cell] = (int)(cell * (p - 1) * (p - 1) * (p - 1));
      }
  std::vector<int> cons((size_t)op->n_constrained);
  if (!cons.empty())
    BP5_CUDA(cudaMemcpyAsync(cons.data(), op->constrained, sizeof(int) * cons.size(), cudaMemcpyDeviceToHost, ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  const int64_t plane = (int64_t)L.nx * L.ny;
  for (int &c : cons) {
    const int k = (int)(c / plane), j = (int)((c - k * plane) / L.nx), i = (int)(c - k * plane - (int64_t)j * L.nx);
    c = (int)blocked_index(L, i, j, k);
  }
  BP5_CUDA(cudaMalloc(&op->blk_desc, sizeof(int) * desc.size()));
  BP5_CUDA(cudaMemcpyAsync(op->blk_desc, desc.data(), sizeof(int) * desc.size(), cudaMemcpyHostToDevice, ctx->stream));
  BP5_CUDA(cudaMalloc(&op->blk_constrained, sizeof(int) * std::max<size_t>(cons.size(), 1)));
  if (!cons.empty())
    BP5_CUDA(cudaMemcpyAsync(op->blk_constrained, cons.data(), sizeof(int) * cons.size(), cudaMemcpyHostToDevice,
                             ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));   // desc and cons live on this stack frame
  op->blk = L;
  return BP5_OK;
}

__global__ void set_constrained_kernel(const int *__restrict__ list, long long n, double value, double *__restrict__ v);
__global__ void hanging_rhs_kernel(BlockGeom g0, BlockGeom g1, const int4 *__restrict__ cells,
                                   const unsigned int *__restrict__ masks, const int *__restrict__ l2g, int pad,
                                   const double *__restrict__ interp, double *__restrict__ b);

int operator_assemble_rhs(bp5_operator_t op, double *b_dev) {
  bp5_context_t ctx = op->ctx;
  const int n = op->n, n3 = n * n * n;
  const BlockGeom g = make_geom(op);
  Tables1D tg;
  make_tables(op->p, BP5_QUAD_GAUSS, tg);   // the reference always assembles with QGauss(p+1), step-64.cu:380
  BP5_CUDA(cudaMemcpyToSymbolAsync(c_tab, &tg, sizeof(Tables1D), 0, cudaMemcpyHostToDevice, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(b_dev, 0, sizeof(double) * (op->n_owned + op->n_ghost), ctx->stream));
  if (op->hanging) {
    BlockGeom g0 = g, g1 = g;
    for (int d = 0; d < 3; ++d) { g0.c0[d] = g1.c0[d] = 0; g1.h[d] = 0.5 * g0.h[d]; }
    const int threads = ((n3 + 31) / 32) * 32;
    hanging_rhs_kernel<<<(unsigned)(op->n_tiles * op->cells_per_tile), threads, sizeof(double) * 8 * n3, ctx->stream>>>(
        g0, g1, static_cast<const int4 *>(op->hanging_cells), op->cell_mask, op->l2g_irr, n3, op->hanging_interp_dev, b_dev);
    BP5_CHECK_LAUNCH();
    if (op->n_constrained > 0) {
      set_constrained_kernel<<<(unsigned)((op->n_constrained + 255) / 256), 256, 0, ctx->stream>>>(op->constrained,
                                                                                                op->n_constrained, 0.0, b_dev);
      BP5_CHECK_LAUNCH();
    }
    ctx->launches += 2;
    BP5_CUDA(cudaMemcpyToSymbolAsync(c_tab, &op->tab, sizeof(Tables1D), 0, cudaMemcpyHostToDevice, ctx->stream));
    BP5_CUDA(cudaStreamSynchronize(ctx->stream));
    return BP5_OK;
  }
  const int ex = op->lc[0] + op->has_hi[0], ey = op->lc[1] + op->has_hi[1], ez = op->lc[2] + op->has_hi[2];
  const int threads = ((n3 + 31) / 32) * 32;
  rhs_kernel<<<(unsigned)((long long)ex * ey * ez), threads, sizeof(double) * 8 * n3, ctx->stream>>>(g, ex, ey, ez, b_dev);
  BP5_CHECK_LAUNCH();
  ctx->launches++;
  // restore the operator's own tables for later setup calls
  BP5_CUDA(cudaMemcpyToSymbolAsync(c_tab, &op->tab, sizeof(Tables1D), 0, cudaMemcpyHostToDevice, ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  return BP5_OK;
}

int operator_export_coefficients(bp5_operator_t op, double *host_out) {
  // internal layout [cell][plane][q] -> reference layout coef[plane][cell][q]
  // (bp5/step-64.cu:108,112), first 6 planes.
  const int n3 = op->n * op->n * op->n;
  const int P = op->metric_planes;
  std::vector<double> tmp((size_t)op->n_tiles * op->tile_doubles);
  BP5_CUDA(cudaMemcpy(tmp.data(), op->metric, sizeof(double) * tmp.size(), cudaMemcpyDeviceToHost));
  std::vector<long long> slot_of;
  cell_slots(op, slot_of);
  for (int64_t c = 0; c < op->n_cells; ++c) {
    const int64_t sl = slot_of[c];   // processing-order slot, see operator_plan_tiles
    const size_t base = (size_t)(sl / op->cells_per_tile) * op->tile_doubles + (size_t)(sl % op->cells_per_tile) * P * n3;
    for (int pl = 0; pl < 6; ++pl)
      std::copy_n(&tmp[base + (size_t)pl * n3], n3, &host_out[((size_t)pl * op->n_cells + c) * n3]);
  }
  return BP5_OK;
}

static int dof_info(bp5_operator_t op, double *xyz_host, int64_t *gidx_host) {
  bp5_context_t ctx = op->ctx;
  const BlockGeom g = make_geom(op);
  const int64_t nloc = op->n_owned + op->n_ghost;
  double *xyz = nullptr; long long *gi = nullptr;
  if (xyz_host) BP5_CUDA(cudaMalloc(&xyz, sizeof(double) * 3 * nloc));
  if (gidx_host) BP5_CUDA(cudaMalloc(&gi, sizeof(long long) * nloc));
  BP5_CUDA(cudaMemcpyToSymbolAsync(c_tab, &op->tab, sizeof(Tables1D), 0, cudaMemcpyHostToDevice, ctx->stream));
  const long long tot = (long long)op->ld[0] * op->ld[1] * op->ld[2];
  dof_info_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, ctx->stream>>>(g, xyz, gi);
  BP5_CHECK_LAUNCH();
  ctx->launches++;
  if (xyz_host) BP5_CUDA(cudaMemcpyAsync(xyz_host, xyz, sizeof(double) * 3 * nloc, cudaMemcpyDeviceToHost, ctx->stream));
  if (gidx_host) BP5_CUDA(cudaMemcpyAsync(gidx_host, gi, sizeof(long long) * nloc, cudaMemcpyDeviceToHost, ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  cudaFree(xyz); cudaFree(gi);
  return BP5_OK;
}
int operator_export_coords(bp5_operator_t op, double *host_out) { return dof_info(op, host_out, nullptr); }
int operator_export_global_indices(bp5_operator_t op, int64_t *host_out) { return dof_info(op, nullptr, host_out); }

// ---------------------------------------------------------------------------
// deal.II-layout geometry for user-written cell functors (CUDAWrappers::MatrixFree::Data as
// the reference's functors index it):
//   inv_jacobian[(d*3+e)*n_cells*pad + cell*pad + q]   bp5/step-64.cu:94-97, fe_evaluation_gl.h:340,365
//   JxW[cell*pad + q]                                   bp5/step-64.cu:109, fe_evaluation_gl.h:299
//   local_to_global[cell*pad + i]                       fe_evaluation_gl.h:118,144
//   q_points[cell*pad + q] (3 doubles each)             step-64/step-64.cu:105-108
// pad = next power of two >= n^3 (padding_length).
// The cells written are those of the sub-lattice (off + stride * i) in each direction, numbered x fastest:
// stride 1, off 0 = all cells in lexicographic order; stride 2 = one of the eight parity colours (cells of one
// colour share no DoF, MatrixFree::AdditionalData::use_coloring, bp5/fe_evaluation_gl.h:176-177).
// inverse Jacobian, JxW and quadrature point of this thread's point of lattice cell (cx, cy, cz) of `g`, written at
// `cell` of the deal.II-layout arrays (whole CTA: cell_jacobian synchronises)
__device__ void write_generic_geometry(const BlockGeom &g, double *sm, int cx, int cy, int cz, long long cell,
                                       long long n_cells, int pad, double *__restrict__ inv_jac,
                                       double *__restrict__ jxw, double *__restrict__ qpts) {
  const int n = g.n, n2 = n * n, n3 = n2 * n;
  const int t = threadIdx.x;
  const int i = t % n, j = (t / n) % n, k = t / n2;
  double J[3][3], xr[3];
  cell_jacobian(g, c_tab.B, c_tab.Dg, sm, cx, cy, cz, J, xr);
  if (t >= n3) return;
  const double det = det3(J), id = 1.0 / det;
  double I[3][3];
  I[0][0] = (J[1][1] * J[2][2] - J[1][2] * J[2][1]) * id;
  I[0][1] = (J[0][2] * J[2][1] - J[0][1] * J[2][2]) * id;
  I[0][2] = (J[0][1] * J[1][2] - J[0][2] * J[1][1]) * id;
  I[1][0] = (J[1][2] * J[2][0] - J[1][0] * J[2][2]) * id;
  I[1][1] = (J[0][0] * J[2][2] - J[0][2] * J[2][0]) * id;
  I[1][2] = (J[0][2] * J[1][0] - J[0][0] * J[1][2]) * id;
  I[2][0] = (J[1][0] * J[2][1] - J[1][1] * J[2][0]) * id;
  I[2][1] = (J[0][1] * J[2][0] - J[0][0] * J[2][1]) * id;
  I[2][2] = (J[0][0] * J[1][1] - J[0][1] * J[1][0]) * id;
  const long long plane = n_cells * pad, at = cell * pad + t;
  for (int d = 0; d < 3; ++d)
    for (int e = 0; e < 3; ++e) inv_jac[(d * 3 + e) * plane + at] = I[d][e];
  jxw[at] = det * c_tab.wq[i] * c_tab.wq[j] * c_tab.wq[k];
  for (int d = 0; d < 3; ++d) qpts[3 * at + d] = xr[d];
}

struct CellLattice { int stride, off[3], dims[3]; };
__global__ void generic_data_kernel(BlockGeom g, CellLattice lat, int pad, unsigned int *__restrict__ l2g,
                                    double *__restrict__ inv_jac, double *__restrict__ jxw, double *__restrict__ qpts) {
  extern __shared__ double sm[];
  const int n = g.n, n2 = n * n, n3 = n2 * n;
  const long long cell = blockIdx.x;
  const long long n_cells = gridDim.x;
  const int lcx = lat.off[0] + lat.stride * (int)(cell % lat.dims[0]);
  const int lcy = lat.off[1] + lat.stride * (int)((cell / lat.dims[0]) % lat.dims[1]);
  const int lcz = lat.off[2] + lat.stride * (int)(cell / ((long long)lat.dims[0] * lat.dims[1]));
  const int t = threadIdx.x;
  const int i = t % n, j = (t / n) % n, k = t / n2;
  if (t < n3) l2g[cell * pad + t] = (unsigned int)local_dof_index(g, lcx * g.p + i, lcy * g.p + j, lcz * g.p + k);
  write_generic_geometry(g, sm, g.c0[0] + lcx, g.c0[1] + lcy, g.c0[2] + lcz, cell, n_cells, pad, inv_jac, jxw, qpts);
}

// arrays of one cell lattice in deal.II's layout; n_cells_out = 0 leaves everything null
static int build_generic_arrays(bp5_operator_t op, const CellLattice &lat, unsigned int **l2g, double **inv_jac,
                                double **jxw, double **qpts, unsigned int **cmask, int64_t *n_cells_out) {
  bp5_context_t ctx = op->ctx;
  const int n = op->n, n3 = n * n * n, pad = op->mf_padding;
  const size_t cells = (size_t)lat.dims[0] * lat.dims[1] * lat.dims[2];
  *n_cells_out = (int64_t)cells;
  if (cells == 0) return BP5_OK;
  BP5_CUDA(cudaMalloc(l2g, sizeof(unsigned int) * cells * pad));
  BP5_CUDA(cudaMalloc(inv_jac, sizeof(double) * 9 * cells * pad));
  BP5_CUDA(cudaMalloc(jxw, sizeof(double) * cells * pad));
  BP5_CUDA(cudaMalloc(qpts, sizeof(double) * 3 * cells * pad));
  BP5_CUDA(cudaMalloc(cmask, sizeof(unsigned int) * cells));
  BP5_CUDA(cudaMemsetAsync(*l2g, 0, sizeof(unsigned int) * cells * pad, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(*inv_jac, 0, sizeof(double) * 9 * cells * pad, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(*jxw, 0, sizeof(double) * cells * pad, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(*qpts, 0, sizeof(double) * 3 * cells * pad, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(*cmask, 0, sizeof(unsigned int) * cells, ctx->stream));   // conforming mesh
  const BlockGeom g = make_geom(op);
  BP5_CUDA(cudaMemcpyToSymbolAsync(c_tab, &op->tab, sizeof(Tables1D), 0, cudaMemcpyHostToDevice, ctx->stream));
  const int threads = ((n3 + 31) / 32) * 32;
  generic_data_kernel<<<(unsigned)cells, threads, sizeof(double) * 8 * n3, ctx->stream>>>(g, lat, pad, *l2g, *inv_jac, *jxw,
                                                                                        *qpts);
  BP5_CHECK_LAUNCH();
  ctx->launches++;
  return BP5_OK;
}

// the same arrays once per parity colour (px, py, pz), colour = px + 2 py + 4 pz
int operator_generic_data_colored(bp5_operator_t op) {
  if (op->mf_colors_built) return BP5_OK;
  int pad = 1;
  while (pad < op->n * op->n * op->n) pad <<= 1;
  op->mf_padding = pad;
  for (int c = 0; c < 8; ++c) {
    CellLattice lat;
    lat.stride = 2;
    for (int d = 0; d < 3; ++d) {
      lat.off[d] = (c >> d) & 1;
      lat.dims[d] = op->lc[d] > lat.off[d] ? (op->lc[d] - lat.off[d] + 1) / 2 : 0;
    }
    int rc = build_generic_arrays(op, lat, &op->mfc_l2g[c], &op->mfc_inv_jacobian[c], &op->mfc_jxw[c], &op->mfc_q_points[c],
                                  &op->mfc_constraint_mask[c], &op->mfc_n_cells[c]);
    if (rc) return rc;
  }
  BP5_CUDA(cudaStreamSynchronize(op->ctx->stream));
  op->mf_colors_built = true;
  return BP5_OK;
}

int operator_generic_data(bp5_operator_t op) {
  if (op->mf_l2g) return BP5_OK;
  bp5_context_t ctx = op->ctx;
  const int n = op->n, n3 = n * n * n;
  int pad = 1;
  while (pad < n3) pad <<= 1;
  op->mf_padding = pad;
  const size_t cells = (size_t)op->n_cells;
  BP5_CUDA(cudaMalloc(&op->mf_l2g, sizeof(unsigned int) * cells * pad));
  BP5_CUDA(cudaMalloc(&op->mf_inv_jacobian, sizeof(double) * 9 * cells * pad));
  BP5_CUDA(cudaMalloc(&op->mf_jxw, sizeof(double) * cells * pad));
  BP5_CUDA(cudaMalloc(&op->mf_q_points, sizeof(double) * 3 * cells * pad));
  BP5_CUDA(cudaMalloc(&op->mf_constraint_mask, sizeof(unsigned int) * cells));
  BP5_CUDA(cudaMemsetAsync(op->mf_l2g, 0, sizeof(unsigned int) * cells * pad, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(op->mf_inv_jacobian, 0, sizeof(double) * 9 * cells * pad, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(op->mf_jxw, 0, sizeof(double) * cells * pad, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(op->mf_q_points, 0, sizeof(double) * 3 * cells * pad, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(op->mf_constraint_mask, 0, sizeof(unsigned int) * cells, ctx->stream));   // conforming mesh
  const BlockGeom g = make_geom(op);
  BP5_CUDA(cudaMemcpyToSymbolAsync(c_tab, &op->tab, sizeof(Tables1D), 0, cudaMemcpyHostToDevice, ctx->stream));
  const int threads = ((n3 + 31) / 32) * 32;
  const CellLattice all{1, {0, 0, 0}, {op->lc[0], op->lc[1], op->lc[2]}};
  generic_data_kernel<<<(unsigned)op->n_cells, threads, sizeof(double) * 8 * n3, ctx->stream>>>(
      g, all, pad, op->mf_l2g, op->mf_inv_jacobian, op->mf_jxw, op->mf_q_points);
  BP5_CHECK_LAUNCH();
  ctx->launches++;
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  return BP5_OK;
}

// ---------------------------------------------------------------------------
// Locally refined meshes with hanging nodes, for the generic functor path -- the `constraint_mask` /
// resolve_hanging_nodes slot of the reference's evaluator (bp5/fe_evaluation_gl.h:88,150,167), which none of its
// meshes exercises.  The coarse cells with indices in [refine_lo, refine_hi) are replaced by their eight children
// (one level: 2:1 balanced by construction).  A child face that lies on a face of an unrefined neighbour carries no
// DoFs of its own: its nodes take the values of the neighbour's face polynomial.
//   numbering   coarse-lattice nodes that belong to an unrefined cell, x fastest; then the nodes of the fine lattice
//               over the refined box that are not hanging, x fastest (the CPU restatement used by the tests numbers the same way)
//   cells       unrefined coarse cells, x fastest; then the children, parents x fastest, child = sx + 2 sy + 4 sz
//   l2g         a local node ON a constrained face holds the PARENT's node with the same local index (which lies on
//               the unrefined neighbour's face); the evaluator turns those values into the child's by 1D
//               interpolations along the face's lines (read) or their transposes (distribute)
//   mask        bit d (0..2): the child's face normal to d on the parent's boundary is constrained;
//               bit 3 + d: the child's position s_d in the parent (selects the face: low if 0, high if 1, and the
//               1D interpolation matrix along d).  Unrefined cells: 0.
// the stored metric of the tuned kernel, cells in the order of the descriptors (= processing order)
__global__ void hanging_metric_kernel(BlockGeom g0, BlockGeom g1, const int4 *__restrict__ cells,
                                      double *__restrict__ metric) {
  extern __shared__ double sm[];
  const int4 c = cells[blockIdx.x];      // one CTA per cell SLOT of the processing order
  if (c.w < 0) return;                   // tile padding
  write_cell_metric(c.w ? g1 : g0, sm, c.x, c.y, c.z, blockIdx.x, metric);
}
// the generic functor path's arrays (deal.II layout), built on first use: geometry per cell, the index tables padded to
// padding_length, the masks
// (one CTA per cell slot; the arrays are compact: cell = slot minus the padding between the two groups of cells)
__global__ void hanging_geometry_kernel(BlockGeom g0, BlockGeom g1, const int4 *__restrict__ cells, int pad,
                                        long long n_first, long long first_padded, long long n_cells,
                                        const int *__restrict__ tables, const unsigned int *__restrict__ slot_mask,
                                        unsigned int *__restrict__ l2g, unsigned int *__restrict__ masks,
                                        double *__restrict__ inv_jac, double *__restrict__ jxw,
                                        double *__restrict__ qpts) {
  extern __shared__ double sm[];
  const long long slot = blockIdx.x;
  const int4 c = cells[slot];
  if (c.w < 0) return;
  const long long cell = slot < first_padded ? slot : slot - (first_padded - n_first);
  const int n3 = g0.n * g0.n * g0.n;
  if ((int)threadIdx.x < n3) l2g[cell * pad + threadIdx.x] = (unsigned int)tables[slot * n3 + threadIdx.x];
  if (threadIdx.x == 0) masks[cell] = slot_mask[slot] & 63u;     // without the stride class
  write_generic_geometry(c.w ? g1 : g0, sm, c.x, c.y, c.z, cell, n_cells, pad, inv_jac, jxw, qpts);
}

int operator_generic_data_hanging(bp5_operator_t op) {
  if (op->mf_l2g) return BP5_OK;
  bp5_context_t ctx = op->ctx;
  const int n3 = op->n * op->n * op->n, pad = op->mf_padding;
  const size_t cells = (size_t)op->n_cells;
  BP5_CUDA(cudaMalloc(&op->mf_l2g, sizeof(unsigned int) * cells * pad));
  BP5_CUDA(cudaMalloc(&op->mf_constraint_mask, sizeof(unsigned int) * cells));
  BP5_CUDA(cudaMalloc(&op->mf_inv_jacobian, sizeof(double) * 9 * cells * pad));
  BP5_CUDA(cudaMalloc(&op->mf_jxw, sizeof(double) * cells * pad));
  BP5_CUDA(cudaMalloc(&op->mf_q_points, sizeof(double) * 3 * cells * pad));
  BP5_CUDA(cudaMemsetAsync(op->mf_l2g, 0, sizeof(unsigned int) * cells * pad, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(op->mf_inv_jacobian, 0, sizeof(double) * 9 * cells * pad, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(op->mf_jxw, 0, sizeof(double) * cells * pad, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(op->mf_q_points, 0, sizeof(double) * 3 * cells * pad, ctx->stream));
  BlockGeom g0 = make_geom(op), g1 = g0;
  for (int d = 0; d < 3; ++d) { g0.c0[d] = g1.c0[d] = 0; g1.h[d] = 0.5 * g0.h[d]; }
  BP5_CUDA(cudaMemcpyToSymbolAsync(c_tab, &op->tab, sizeof(Tables1D), 0, cudaMemcpyHostToDevice, ctx->stream));
  const int threads = ((n3 + 31) / 32) * 32;
  const long long padded = op->n_tiles * op->cells_per_tile;
  hanging_geometry_kernel<<<(unsigned)padded, threads, sizeof(double) * 8 * n3, ctx->stream>>>(
      g0, g1, static_cast<const int4 *>(op->hanging_cells), pad, op->n_boundary_cells,
      op->n_boundary_tiles * op->cells_per_tile, op->n_cells, op->l2g_irr, op->cell_mask, op->mf_l2g,
      op->mf_constraint_mask, op->mf_inv_jacobian, op->mf_jxw, op->mf_q_points);
  BP5_CHECK_LAUNCH();
  ctx->launches++;
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  return BP5_OK;
}

static void host_map_point(const bp5_problem_t &pr, const double *x, double *y) {
  if (pr.deformation == 0) { y[0] = x[0]; y[1] = x[1]; y[2] = x[2]; return; }
  double s = 1.0;
  for (int d = 0; d < 3; ++d) s *= sin(M_PI * (x[d] - pr.lower[d]) / (pr.upper[d] - pr.lower[d]));
  for (int d = 0; d < 3; ++d) y[d] = x[d] + pr.deformation_eps * (pr.upper[d] - pr.lower[d]) * s;
}

int operator_setup_hanging(bp5_operator_t op) {
  bp5_context_t ctx = op->ctx;
  const bp5_problem_t &pr = op->prob;
  const int p = op->p, n = op->n, n3 = n * n * n;
  const int *c = pr.cells, *r0 = pr.refine_lo, *r1 = pr.refine_hi;
  auto in_box = [&](int i, int j, int k) {
    return i >= r0[0] && i < r1[0] && j >= r0[1] && j < r1[1] && k >= r0[2] && k < r1[2];
  };
  // ---- numbering
  const int64_t nc[3] = {(int64_t)c[0] * p + 1, (int64_t)c[1] * p + 1, (int64_t)c[2] * p + 1};
  const int64_t nf[3] = {2ll * (r1[0] - r0[0]) * p + 1, 2ll * (r1[1] - r0[1]) * p + 1, 2ll * (r1[2] - r0[2]) * p + 1};
  const int64_t f0[3] = {2ll * r0[0] * p, 2ll * r0[1] * p, 2ll * r0[2] * p};
  BP5_REQUIRE(nc[0] * nc[1] * nc[2] + nf[0] * nf[1] * nf[2] < (int64_t)2147483647, "mesh too large for 32-bit indices");
  std::vector<int> coarse_id((size_t)(nc[0] * nc[1] * nc[2]), -1), fine_id((size_t)(nf[0] * nf[1] * nf[2]), -1);
  std::vector<int> cons;
  std::vector<double> &X = op->hanging_coords;
  X.clear();
  const double h0[3] = {(pr.upper[0] - pr.lower[0]) / c[0], (pr.upper[1] - pr.lower[1]) / c[1],
                        (pr.upper[2] - pr.lower[2]) / c[2]};
  // node k of a lattice with `cells` cells of size h: the cell that holds it and its local index
  auto lattice_point = [&](const int64_t k[3], const int cells_d[3], double scale, double *y) {
    double x[3];
    for (int d = 0; d < 3; ++d) {
      const int i = (int)std::min<int64_t>(k[d] / p, cells_d[d] - 1);
      x[d] = pr.lower[d] + h0[d] * scale * (i + op->tab.xi[k[d] - (int64_t)i * p]);
    }
    host_map_point(pr, x, y);
  };
  int N = 0;
  for (int64_t kz = 0; kz < nc[2]; ++kz)
    for (int64_t ky = 0; ky < nc[1]; ++ky)
      for (int64_t kx = 0; kx < nc[0]; ++kx) {
        const int64_t k[3] = {kx, ky, kz};
        int lo[3], hi[3];
        for (int d = 0; d < 3; ++d) {
          hi[d] = (int)std::min<int64_t>(k[d] / p, c[d] - 1);
          lo[d] = (k[d] % p == 0 && k[d] > 0) ? (int)(k[d] / p) - 1 : hi[d];
        }
        bool used = false;
        for (int iz = lo[2]; iz <= hi[2]; ++iz)
          for (int iy = lo[1]; iy <= hi[1]; ++iy)
            for (int ix = lo[0]; ix <= hi[0]; ++ix) used |= !in_box(ix, iy, iz);
        if (!used) continue;
        coarse_id[(size_t)(kx + nc[0] * (ky + nc[1] * kz))] = N;
        if (kx == 0 || kx == nc[0] - 1 || ky == 0 || ky == nc[1] - 1 || kz == 0 || kz == nc[2] - 1) cons.push_back(N);
        double y[3];
        lattice_point(k, c, 1.0, y);
        X.insert(X.end(), y, y + 3);
        ++N;
      }
  const int c2[3] = {2 * c[0], 2 * c[1], 2 * c[2]};
  for (int64_t fz = 0; fz < nf[2]; ++fz)
    for (int64_t fy = 0; fy < nf[1]; ++fy)
      for (int64_t fx = 0; fx < nf[0]; ++fx) {
        const int64_t f[3] = {fx, fy, fz};
        bool hanging = false, boundary = false;
        int64_t k[3];
        for (int d = 0; d < 3; ++d) {
          hanging |= (f[d] == 0 && r0[d] > 0) || (f[d] == nf[d] - 1 && r1[d] < c[d]);
          k[d] = f0[d] + f[d];
          boundary |= k[d] == 0 || k[d] == 2ll * c[d] * p;
        }
        if (hanging) continue;
        fine_id[(size_t)(fx + nf[0] * (fy + nf[1] * fz))] = N;
        if (boundary) cons.push_back(N);
        double y[3];
        lattice_point(k, c2, 0.5, y);
        X.insert(X.end(), y, y + 3);
        ++N;
      }
  // ---- cells
  const int64_t n_box = (int64_t)(r1[0] - r0[0]) * (r1[1] - r0[1]) * (r1[2] - r0[2]);
  const int64_t n_cells = (int64_t)c[0] * c[1] * c[2] - n_box + 8 * n_box;
  int pad = 1;
  while (pad < n3) pad <<= 1;
  op->mf_padding = pad;
  std::vector<int> l2g((size_t)n_cells * n3, 0);      // [cell][n3]: the tuned kernel's index tables
  std::vector<unsigned int> mask((size_t)n_cells, 0u);
  std::vector<int4> desc((size_t)n_cells);
  int64_t cell = 0;
  for (int cz = 0; cz < c[2]; ++cz)
    for (int cy = 0; cy < c[1]; ++cy)
      for (int cx = 0; cx < c[0]; ++cx) {
        if (in_box(cx, cy, cz)) continue;
        for (int t = 0; t < n3; ++t) {
          const int64_t kx = (int64_t)cx * p + t % n, ky = (int64_t)cy * p + (t / n) % n, kz = (int64_t)cz * p + t / (n * n);
          l2g[(size_t)cell * n3 + t] = coarse_id[(size_t)(kx + nc[0] * (ky + nc[1] * kz))];
        }
        desc[(size_t)cell] = make_int4(cx, cy, cz, 0);
        ++cell;
      }
  for (int pz = r0[2]; pz < r1[2]; ++pz)
    for (int py = r0[1]; py < r1[1]; ++py)
      for (int px = r0[0]; px < r1[0]; ++px)
        for (int s = 0; s < 8; ++s) {
          const int par[3] = {px, py, pz}, sd[3] = {s & 1, (s >> 1) & 1, (s >> 2) & 1};
          unsigned int m = 0;
          int face[3];   // local index of the constrained face's plane, -1: not constrained
          for (int d = 0; d < 3; ++d) {
            const bool con = sd[d] == 0 ? (par[d] == r0[d] && r0[d] > 0) : (par[d] == r1[d] - 1 && r1[d] < c[d]);
            face[d] = con ? (sd[d] ? p : 0) : -1;
            if (con) m |= 1u << d;
            m |= (unsigned int)sd[d] << (3 + d);
          }
          if ((m & 7u) == 0) m = 0;          // nothing to resolve: plain cell
          mask[(size_t)cell] = m;
          for (int t = 0; t < n3; ++t) {
            const int a[3] = {t % n, (t / n) % n, t / (n * n)};
            const bool on_face = a[0] == face[0] || a[1] == face[1] || a[2] == face[2];
            int id;
            if (on_face) {
              const int64_t kx = (int64_t)px * p + a[0], ky = (int64_t)py * p + a[1], kz = (int64_t)pz * p + a[2];
              id = coarse_id[(size_t)(kx + nc[0] * (ky + nc[1] * kz))];
            } else {
              const int64_t fx = (2ll * px + sd[0]) * p + a[0] - f0[0], fy = (2ll * py + sd[1]) * p + a[1] - f0[1],
                            fz = (2ll * pz + sd[2]) * p + a[2] - f0[2];
              id = fine_id[(size_t)(fx + nf[0] * (fy + nf[1] * fz))];
            }
            BP5_REQUIRE(id >= 0, "internal error: cell node without a DoF on the locally refined mesh");
            l2g[(size_t)cell * n3 + t] = id;
          }
          desc[(size_t)cell] = make_int4(2 * px + sd[0], 2 * py + sd[1], 2 * pz + sd[2], 1);
          ++cell;
        }
  BP5_REQUIRE(cell == n_cells, "internal error: cell count of the locally refined mesh");
  // ---- sizes, Dirichlet set, 1D parent-to-child interpolation
  op->n_owned = N; op->n_ghost = 0; op->n_global = N; op->n_cells = n_cells;
  op->hanging = true;
  std::sort(cons.begin(), cons.end());
  op->n_constrained = (int64_t)cons.size();
  BP5_CUDA(cudaMalloc(&op->constrained, sizeof(int) * std::max<size_t>(cons.size(), 1)));
  BP5_CUDA(cudaMemcpyAsync(op->constrained, cons.data(), sizeof(int) * cons.size(), cudaMemcpyHostToDevice, ctx->stream));
  parent_child_interp(op->tab, op->hanging_interp);
  // ---- the tuned kernel's view of the same cells (apply.cuh, HANG).
  // The numbering is piecewise lexicographic: a cell without a constrained face whose n^3 indices are
  // base + i + j sy + k sz gets the affine descriptor (base >= 0) and the class of its stride pair (at most 8 classes,
  // cell_mask bits 8..10).  The others -- children with a constrained face, cells across a seam of the numbering --
  // go through an index table (cell_base < 0 selects table -(base + 1) of l2g_irr) and come FIRST in the processing
  // order, padded to whole tiles like the boundary cells of a partitioned block: tiles [0, n_boundary_tiles) run the
  // kernel with the constraint exchange (HANG = 1), the rest the one without (HANG = 2).
  std::vector<int> cls((size_t)n_cells, -1), base_of((size_t)n_cells, 0);
  int n_classes = 0;
  int64_t n_first = 0;
  for (int64_t cI = 0; cI < n_cells; ++cI) {
    bool affine = mask[(size_t)cI] == 0;
    const int *id = &l2g[(size_t)cI * n3];
    const int b0 = id[0], sy = id[n] - b0, sz = id[n * n] - b0;
    for (int t = 0; t < n3 && affine; ++t) affine = id[t] == b0 + t % n + sy * ((t / n) % n) + sz * (t / (n * n));
    if (affine) {
      int cl = 0;
      while (cl < n_classes && !(op->hang_sy[cl] == sy && op->hang_sz[cl] == sz)) ++cl;
      if (cl == n_classes && n_classes < 8) { op->hang_sy[cl] = sy; op->hang_sz[cl] = sz; ++n_classes; }
      if (cl < n_classes) { cls[(size_t)cI] = cl; base_of[(size_t)cI] = b0; }
    }
    if (cls[(size_t)cI] < 0) ++n_first;
  }
  op->n_boundary_cells = n_first;
  op->hanging_affine_cells = n_cells - n_first;
  {
    const int rc = apply_choose(op);     // cells per tile, tile plan (operator_plan_tiles), kernel name
    if (rc != BP5_OK) return rc;
  }
  const int64_t padded = op->n_tiles * op->cells_per_tile, first_padded = op->n_boundary_tiles * op->cells_per_tile;
  int4 *desc_dev = nullptr;
  {
    std::vector<int> base((size_t)padded, INT_MIN), table((size_t)padded * n3, 0);
    std::vector<unsigned int> slot_mask((size_t)padded, 0u);
    std::vector<int4> slot_desc((size_t)padded, make_int4(0, 0, 0, -1));     // w < 0: tile padding
    int64_t next_first = 0, next_rest = first_padded;
    for (int64_t cI = 0; cI < n_cells; ++cI) {
      const bool first = cls[(size_t)cI] < 0;
      const int64_t slot = first ? next_first++ : next_rest++;
      base[(size_t)slot] = first ? -(int)slot - 1 : base_of[(size_t)cI];
      slot_mask[(size_t)slot] = first ? mask[(size_t)cI] : (unsigned int)cls[(size_t)cI] << 8;
      slot_desc[(size_t)slot] = desc[(size_t)cI];
      std::copy_n(&l2g[(size_t)cI * n3], n3, &table[(size_t)slot * n3]);
    }
    op->n_irregular = padded;
    BP5_CUDA(cudaMalloc(&desc_dev, sizeof(int4) * padded));
    op->hanging_cells = desc_dev;      // owned by the operator from here on (kept for assemble_rhs, l2_norm, ...)
    BP5_CUDA(cudaMalloc(&op->cell_base, sizeof(int) * padded));
    BP5_CUDA(cudaMalloc(&op->cell_mask, sizeof(unsigned int) * padded));
    BP5_CUDA(cudaMalloc(&op->l2g_irr, sizeof(int) * table.size()));
    BP5_CUDA(cudaMemcpyAsync(desc_dev, slot_desc.data(), sizeof(int4) * padded, cudaMemcpyHostToDevice, ctx->stream));
    BP5_CUDA(cudaMemcpyAsync(op->cell_base, base.data(), sizeof(int) * padded, cudaMemcpyHostToDevice, ctx->stream));
    BP5_CUDA(cudaMemcpyAsync(op->cell_mask, slot_mask.data(), sizeof(unsigned int) * padded, cudaMemcpyHostToDevice, ctx->stream));
    BP5_CUDA(cudaMemcpyAsync(op->l2g_irr, table.data(), sizeof(int) * table.size(), cudaMemcpyHostToDevice, ctx->stream));
    const size_t mbytes = sizeof(double) * op->n_tiles * op->tile_doubles;
    BP5_CUDA(cudaMalloc(&op->metric, mbytes));
    BP5_CUDA(cudaMemsetAsync(op->metric, 0, mbytes, ctx->stream));
    BP5_CUDA(cudaStreamSynchronize(ctx->stream));     // the host vectors above go out of scope
  }
  BlockGeom g0 = make_geom(op), g1 = g0;
  for (int d = 0; d < 3; ++d) { g0.c0[d] = g1.c0[d] = 0; g1.h[d] = 0.5 * g0.h[d]; }
  BP5_CUDA(cudaMemcpyToSymbolAsync(c_tab, &op->tab, sizeof(Tables1D), 0, cudaMemcpyHostToDevice, ctx->stream));
  const int threads = ((n3 + 31) / 32) * 32;
  hanging_metric_kernel<<<(unsigned)padded, threads, sizeof(double) * 8 * n3, ctx->stream>>>(g0, g1, desc_dev, op->metric);
  BP5_CHECK_LAUNCH();
  ctx->launches++;
  BP5_CUDA(cudaMalloc(&op->hanging_interp_dev, sizeof(double) * 2 * kMaxN * kMaxN));
  BP5_CUDA(cudaMemcpyAsync(op->hanging_interp_dev, op->hanging_interp, sizeof(double) * 2 * kMaxN * kMaxN,
                           cudaMemcpyHostToDevice, ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  return BP5_OK;
}

// b_i = int phi_i with QGauss(p+1) on a locally refined mesh (c_tab must hold the GAUSS tables): per cell the local
// integrals, the transposed hanging-node constraints (what constraints.distribute_local_to_global does at
// bp5/step-64.cu:411), scatter-add.  One thread per local node.
__global__ void hanging_rhs_kernel(BlockGeom g0, BlockGeom g1, const int4 *__restrict__ cells,
                                   const unsigned int *__restrict__ masks, const int *__restrict__ l2g, int pad,
                                   const double *__restrict__ interp, double *__restrict__ b) {
  extern __shared__ double sm[];
  const int4 c = cells[blockIdx.x];      // one CTA per cell slot
  if (c.w < 0) return;                   // tile padding
  const BlockGeom &g = c.w ? g1 : g0;
  const int n = g.n, n2 = n * n, n3 = n2 * n;
  const int t = threadIdx.x;
  const int i = t % n, j = (t / n) % n, k = t / n2;
  double J[3][3], xr[3];
  cell_jacobian(g, c_tab.B, c_tab.Dg, sm, c.x, c.y, c.z, J, xr);
  double *w0 = sm, *w1 = sm + n3;
  if (t < n3) w0[t] = det3(J) * c_tab.wq[i] * c_tab.wq[j] * c_tab.wq[k];
  __syncthreads();
  if (t < n3) { double s = 0; for (int m = 0; m < n; ++m) s += c_tab.B[m * n + i] * w0[(k * n + j) * n + m]; w1[t] = s; }
  __syncthreads();
  if (t < n3) { double s = 0; for (int m = 0; m < n; ++m) s += c_tab.B[m * n + j] * w1[(k * n + m) * n + i]; w0[t] = s; }
  __syncthreads();
  if (t < n3) { double s = 0; for (int m = 0; m < n; ++m) s += c_tab.B[m * n + k] * w0[(m * n + j) * n + i]; w1[t] = s; }
  __syncthreads();
  // transposed constraints, direction by direction (mask uniform per cell)
  const unsigned int mask = masks[blockIdx.x] & 63u;
  if (mask != 0) {
    const int pos[3] = {i, j, k}, stride[3] = {1, n, n2};
    bool on_face[3];
    for (int d = 0; d < 3; ++d) on_face[d] = ((mask >> d) & 1u) && pos[d] == (((mask >> (3 + d)) & 1u) ? n - 1 : 0);
    for (int d = 0; d < 3; ++d) {
      if (((mask & 7u) & ~(1u << d)) == 0) continue;
      const double *M = interp + ((mask >> (3 + d)) & 1u) * kMaxN * kMaxN;
      double v = 0.0;
      const bool in_face = t < n3 && (on_face[(d + 1) % 3] || on_face[(d + 2) % 3]);
      if (t < n3) {
        v = w1[t];
        if (in_face) {
          v = 0.0;
          const int base = t - pos[d] * stride[d];
          for (int m = 0; m < n; ++m) v += M[m * n + pos[d]] * w1[base + m * stride[d]];
        }
      }
      __syncthreads();
      if (t < n3) w1[t] = v;
      __syncthreads();
    }
  }
  if (t < n3) atomicAdd(&b[l2g[(long long)blockIdx.x * pad + t]], w1[t]);
}

// ---------------------------------------------------------------------------
// Diagonal of the operator, for a Jacobi preconditioner in the DiagonalMatrix slot of the solver
// (bp5/step-64.cu:428-432 passes a vector of ones; SURVEY 8f.2).  Per cell and node i:
//   sum_q  grad phi_i(q)^T G(q) grad phi_i(q)  (+ a JxW phi_i(q)^2 for Helmholtz)
// evaluated directly from the stored metric (one CTA per cell slot, one thread per node; set-up cost only),
// accumulated over the cells sharing the node; Dirichlet rows are 1 (vmult copies them, bp5/step-64.cu:275).
// Locally refined meshes: `words` is the per-slot mask word (constraint bits 0..5, stride class bits 8..10) and
// class_sy / class_sz the stride classes; the positions on a constrained face of a child are left to
// hanging_diagonal_kernel.
struct DiagHanging { const unsigned int *words; int class_sy[8], class_sz[8]; };
__device__ __forceinline__ bool on_constrained_face(unsigned int mask, int n, int a, int b, int c) {
  const int pos[3] = {a, b, c};
  bool r = false;
  for (int d = 0; d < 3; ++d) r |= ((mask >> d) & 1u) && pos[d] == (((mask >> (3 + d)) & 1u) ? n - 1 : 0);
  return r;
}
__global__ void diagonal_kernel(int n, int planes, int cpt, long long tile_doubles, const int *__restrict__ cell_base,
                                const int *__restrict__ l2g_irr, const double *__restrict__ metric, int sy, int sz,
                                DiagHanging hang, double *__restrict__ diag) {
  const int n2 = n * n, n3 = n2 * n;
  const long long slot = blockIdx.x;
  const int base = cell_base[slot];
  const int t = threadIdx.x;
  if (base == INT_MIN || t >= n3) return;
  const int a = t % n, b = (t / n) % n, c = t / n2;
  if (hang.words != nullptr) {
    const unsigned int w = hang.words[slot];
    if (on_constrained_face(w & 63u, n, a, b, c)) return;
    sy = hang.class_sy[(w >> 8) & 7u]; sz = hang.class_sz[(w >> 8) & 7u];
  }
  const double *G = metric + (slot / cpt) * tile_doubles + (slot % cpt) * (long long)planes * n3;
  double s = 0.0;
  for (int qz = 0; qz < n; ++qz) {
    const double bz = c_tab.B[qz * n + c], dz = c_tab.Dg[qz * n + c];
    for (int qy = 0; qy < n; ++qy) {
      const double by = c_tab.B[qy * n + b], dy = c_tab.Dg[qy * n + b];
      if (bz == 0.0 && dz == 0.0) continue;
      for (int qx = 0; qx < n; ++qx) {
        const double bx = c_tab.B[qx * n + a], dx = c_tab.Dg[qx * n + a];
        const double gx = dx * by * bz, gy = bx * dy * bz, gz = bx * by * dz;
        if (gx == 0.0 && gy == 0.0 && gz == 0.0 && planes == 6) continue;
        const int q = (qz * n + qy) * n + qx;
        s += G[q] * gx * gx + G[n3 + q] * gy * gy + G[2 * n3 + q] * gz * gz +
             2.0 * (G[3 * n3 + q] * gx * gy + G[4 * n3 + q] * gx * gz + G[5 * n3 + q] * gy * gz);
        if (planes == 7) { const double v = bx * by * bz; s += G[6 * n3 + q] * v * v; }
      }
    }
  }
  const long long idx = base >= 0 ? (long long)base + a + (long long)b * sy + (long long)c * sz
                                  : (long long)l2g_irr[(long long)(-(base + 1)) * n3 + t];
  atomicAdd(&diag[idx], s);
}

// Diagonal entries that come through hanging-node constraints: the coarse DoF j in slot t0 of a constrained child face
// contributes c_j^T K c_j, c_j = (constraint resolution) e_t0 = the trace of j's basis function on the child's nodes.
// One CTA per (slot of the first tile group, local position t0), one thread per node / quadrature point:
// resolve the unit vector, interpolate to the quadrature points, collocation gradient, the quadratic form
// sum_q grad^T G grad (+ mass term) -- no transposes needed.
__global__ void hanging_diagonal_kernel(int n, int planes, int cpt, long long tile_doubles,
                                        const unsigned int *__restrict__ words, const int *__restrict__ tables,
                                        const double *__restrict__ metric, const double *__restrict__ interp,
                                        double *__restrict__ diag) {
  extern __shared__ double sm[];
  const int n2 = n * n, n3 = n2 * n;
  const long long slot = blockIdx.x / n3;
  const int t0 = (int)(blockIdx.x % n3);
  const unsigned int mask = words[slot] & 63u;
  if (mask == 0 || !on_constrained_face(mask, n, t0 % n, (t0 / n) % n, t0 / n2)) return;     // uniform per CTA
  double *v = sm, *w = sm + n3, *red = sm + 2 * n3;
  const int t = threadIdx.x;
  const int pos[3] = {t % n, (t / n) % n, t / n2}, stride[3] = {1, n, n2};
  if (t < n3) v[t] = t == t0 ? 1.0 : 0.0;
  __syncthreads();
  for (int d = 0; d < 3; ++d) {          // forward constraint resolution, direction by direction
    if (((mask & 7u) & ~(1u << d)) == 0) continue;
    const double *M = interp + ((mask >> (3 + d)) & 1u) * kMaxN * kMaxN;
    double val = 0.0;
    if (t < n3) {
      val = v[t];
      bool in_face = false;
      for (int e = 1; e <= 2; ++e) {
        const int o = (d + e) % 3;
        in_face |= ((mask >> o) & 1u) && pos[o] == (((mask >> (3 + o)) & 1u) ? n - 1 : 0);
      }
      if (in_face) {
        val = 0.0;
        const int base = t - pos[d] * stride[d];
        for (int m = 0; m < n; ++m) val += M[pos[d] * n + m] * v[base + m * stride[d]];
      }
    }
    __syncthreads();
    if (t < n3) v[t] = val;
    __syncthreads();
  }
  // values at the quadrature points: B along x, y, z (v -> w -> v -> w)
  for (int d = 0; d < 3; ++d) {
    double *src = (d & 1) ? w : v, *dst = (d & 1) ? v : w;
    if (t < n3) {
      double sum = 0.0;
      const int base = t - pos[d] * stride[d];
      for (int m = 0; m < n; ++m) sum += c_tab.B[pos[d] * n + m] * src[base + m * stride[d]];
      dst[t] = sum;
    }
    __syncthreads();
  }
  double contrib = 0.0;
  if (t < n3) {
    const double *uq = w;                  // after three passes the values sit in w
    double g[3];
    for (int d = 0; d < 3; ++d) {
      double sum = 0.0;
      const int base = t - pos[d] * stride[d];
      for (int m = 0; m < n; ++m) sum += c_tab.Dt[pos[d] * n + m] * uq[base + m * stride[d]];
      g[d] = sum;
    }
    const double *G = metric + (slot / cpt) * tile_doubles + (slot % cpt) * (long long)planes * n3;
    contrib = G[t] * g[0] * g[0] + G[n3 + t] * g[1] * g[1] + G[2 * n3 + t] * g[2] * g[2] +
              2.0 * (G[3 * n3 + t] * g[0] * g[1] + G[4 * n3 + t] * g[0] * g[2] + G[5 * n3 + t] * g[1] * g[2]);
    if (planes == 7) contrib += G[6 * n3 + t] * uq[t] * uq[t];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
  if ((t & 31) == 0) red[t >> 5] = contrib;
  __syncthreads();
  if (t == 0) {
    double sum = 0.0;
    for (int wI = 0; wI < (int)(blockDim.x + 31) / 32; ++wI) sum += red[wI];
    atomicAdd(&diag[tables[slot * n3 + t0]], sum);
  }
}

__global__ void set_constrained_kernel(const int *__restrict__ list, long long n, double value, double *__restrict__ v) {
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (t < n) v[list[t]] = value;
}

__global__ void reciprocal_kernel(double *__restrict__ v, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    v[i] = 1.0 / v[i];
}

int operator_diagonal(bp5_operator_t op, double *diag_dev, bool invert) {
  bp5_context_t ctx = op->ctx;
  if (!op->metric) { set_error("the diagonal needs the stored metric (geometry mode BP5_GEOM_STORED)"); return BP5_ERR_UNSUPPORTED; }
  if (invert && op->n_ghost > 0) {
    set_error("partitioned mesh: compress(add) the diagonal over the blocks first, then invert it");
    return BP5_ERR_UNSUPPORTED;
  }
  const int n = op->n, n3 = n * n * n;
  BP5_CUDA(cudaMemcpyToSymbolAsync(c_tab, &op->tab, sizeof(Tables1D), 0, cudaMemcpyHostToDevice, ctx->stream));
  BP5_CUDA(cudaMemsetAsync(diag_dev, 0, sizeof(double) * (op->n_owned + op->n_ghost), ctx->stream));
  const long long slots = op->n_tiles * op->cells_per_tile;
  const int threads = ((n3 + 31) / 32) * 32;
  DiagHanging hang{};
  if (op->hanging) {
    hang.words = op->cell_mask;
    for (int cl = 0; cl < 8; ++cl) { hang.class_sy[cl] = op->hang_sy[cl]; hang.class_sz[cl] = op->hang_sz[cl]; }
  }
  diagonal_kernel<<<(unsigned)slots, threads, 0, ctx->stream>>>(n, op->metric_planes, op->cells_per_tile, op->tile_doubles,
                                                              op->cell_base, op->l2g_irr, op->metric, op->od[0],
                                                              op->od[0] * op->od[1], hang, diag_dev);
  BP5_CHECK_LAUNCH();
  ctx->launches++;
  if (op->hanging && op->n_boundary_tiles > 0) {
    // the constrained faces of the children: all of them sit in the first tile group
    const long long first_slots = op->n_boundary_tiles * op->cells_per_tile;
    BP5_REQUIRE(first_slots * n3 < (long long)2147483647, "too many constrained cells for one launch");
    hanging_diagonal_kernel<<<(unsigned)(first_slots * n3), threads, sizeof(double) * (2 * n3 + 32), ctx->stream>>>(
        n, op->metric_planes, op->cells_per_tile, op->tile_doubles, op->cell_mask, op->l2g_irr, op->metric,
        op->hanging_interp_dev, diag_dev);
    BP5_CHECK_LAUNCH();
    ctx->launches++;
  }
  if (op->n_constrained > 0) {
    set_constrained_kernel<<<(unsigned)((op->n_constrained + 255) / 256), 256, 0, ctx->stream>>>(op->constrained,
                                                                                              op->n_constrained, 1.0, diag_dev);
    BP5_CHECK_LAUNCH();
    ctx->launches++;
  }
  if (invert) {
    reciprocal_kernel<<<148 * 8, 256, 0, ctx->stream>>>(diag_dev, op->n_owned);
    BP5_CHECK_LAUNCH();
    ctx->launches++;
  }
  return BP5_OK;
}

// ---------------------------------------------------------------------------
// ||u||_L2^2 of the finite element function with QGauss(p+2), this block's cells
// (VectorTools::integrate_difference(..., L2_norm) with a zero reference in output_results,
// bp5/step-64.cu:604-615, step-64/step-64.cu:590-601).  One CTA per cell, one thread per quadrature point;
// values and the Jacobian of the degree-p mapping are evaluated directly (not sum-factorised: this runs
// once per solve).  Per-cell norms are rounded to float like the reference's Vector<float> cellwise_norm and
// added in a fixed order.
struct L2Tables {
  int nq;
  double B[(kMaxN + 1) * kMaxN];    // B[q][i] = phi_i(x_q), x_q Gauss(p+2) points
  double D[(kMaxN + 1) * kMaxN];    // phi_i'(x_q)
  double w[kMaxN + 1];
};

// Locally refined meshes (hang.cells != nullptr): one CTA per cell SLOT; the cell's lattice position and level, its
// index table and constraint mask come from the descriptors of operator_setup_hanging, and the hanging-node constraints
// are resolved on the gathered values (forward interpolation, direction by direction) before the quadrature.
struct L2Hanging {
  const int4 *cells; const int *tables; const unsigned int *masks; const double *interp; double half[3];
};
__global__ void l2_norm_kernel(BlockGeom g, L2Tables tb, L2Hanging hang, const double *__restrict__ u,
                               double *__restrict__ partial) {
  extern __shared__ double sm[];
  const int n = g.n, n2 = n * n, n3 = n2 * n, nq = tb.nq;
  double *U = sm, *X = sm + n3;                      // X[3][n3]
  double *red = X + 3 * n3;                          // [32]
  const long long cell = blockIdx.x;
  int lcx = cell % g.lc[0], lcy = (cell / g.lc[0]) % g.lc[1], lcz = cell / ((long long)g.lc[0] * g.lc[1]);
  double h[3] = {g.h[0], g.h[1], g.h[2]};
  unsigned int mask = 0;
  if (hang.cells != nullptr) {
    const int4 d = hang.cells[cell];
    if (d.w < 0) { if (threadIdx.x == 0) partial[cell] = 0.0; return; }     // tile padding
    lcx = d.x; lcy = d.y; lcz = d.z;
    if (d.w) { h[0] = hang.half[0]; h[1] = hang.half[1]; h[2] = hang.half[2]; }
    mask = hang.masks[cell] & 63u;
  }
  const int c[3] = {g.c0[0] + lcx, g.c0[1] + lcy, g.c0[2] + lcz};
  for (int t = threadIdx.x; t < n3; t += blockDim.x) {
    const int loc[3] = {t % n, (t / n) % n, t / n2};
    U[t] = hang.cells != nullptr ? u[hang.tables[cell * n3 + t]]
                                 : u[local_dof_index(g, lcx * g.p + loc[0], lcy * g.p + loc[1], lcz * g.p + loc[2])];
    double x[3], y[3];
    for (int d = 0; d < 3; ++d) x[d] = g.lo[d] + h[d] * (c[d] + c_tab.xi[loc[d]]);
    map_point(g, x, y);
    for (int d = 0; d < 3; ++d) X[d * n3 + t] = y[d];
  }
  __syncthreads();
  if (mask != 0) {      // uniform per CTA
    const int stride[3] = {1, n, n2};
    for (int d = 0; d < 3; ++d) {
      if (((mask & 7u) & ~(1u << d)) == 0) continue;
      const double *M = hang.interp + ((mask >> (3 + d)) & 1u) * kMaxN * kMaxN;
      double v[2] = {0.0, 0.0};       // blockDim.x >= n3 / 2 always (threads = (p+2)^3 rounded up)
      int slot = 0;
      for (int t = threadIdx.x; t < n3; t += blockDim.x, ++slot) {
        const int pos[3] = {t % n, (t / n) % n, t / n2};
        bool in_face = false;
        for (int e = 1; e <= 2; ++e) {
          const int o = (d + e) % 3;
          in_face |= ((mask >> o) & 1u) && pos[o] == (((mask >> (3 + o)) & 1u) ? n - 1 : 0);
        }
        double val = U[t];
        if (in_face) {
          val = 0.0;
          const int base = t - pos[d] * stride[d];
          for (int m = 0; m < n; ++m) val += M[pos[d] * n + m] * U[base + m * stride[d]];
        }
        v[slot] = val;
      }
      __syncthreads();
      slot = 0;
      for (int t = threadIdx.x; t < n3; t += blockDim.x, ++slot) U[t] = v[slot];
      __syncthreads();
    }
  }
  double contrib = 0.0;
  const int t = threadIdx.x;
  if (t < nq * nq * nq) {
    const int qx = t % nq, qy = (t / nq) % nq, qz = t / (nq * nq);
    double val = 0.0, J[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    for (int k = 0; k < n; ++k) {
      const double bz = tb.B[qz * n + k], dz = tb.D[qz * n + k];
      for (int j = 0; j < n; ++j) {
        const double by = tb.B[qy * n + j], dy = tb.D[qy * n + j];
        for (int i = 0; i < n; ++i) {
          const double bx = tb.B[qx * n + i], dx = tb.D[qx * n + i];
          const int a = (k * n + j) * n + i;
          val += bx * by * bz * U[a];
          for (int d = 0; d < 3; ++d) {
            const double xd = X[d * n3 + a];
            J[d][0] += dx * by * bz * xd; J[d][1] += bx * dy * bz * xd; J[d][2] += bx * by * dz * xd;
          }
        }
      }
    }
    contrib = val * val * det3(J) * tb.w[qx] * tb.w[qy] * tb.w[qz];
  }
  // block sum, fixed order
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
  if ((t & 31) == 0) red[t >> 5] = contrib;
  __syncthreads();
  if (t == 0) {
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) s += red[w];
    // the reference stores the per-cell norms in a Vector<float> before compute_global_error squares and adds
    // them (bp5/step-64.cu:603-613): same rounding here, so the printed norm agrees to the last digit
    const float cell_norm = (float)sqrt(fmax(s, 0.0));
    partial[cell] = (double)cell_norm * (double)cell_norm;
  }
}

__global__ void sum_in_order_kernel(const double *__restrict__ partial, long long n, double *__restrict__ out) {
  __shared__ double sh[256];
  double s = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) s += partial[i];
  sh[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) { double t = 0.0; for (int i = 0; i < 256; ++i) t += sh[i]; *out = t; }
}

int operator_l2_norm_sqr(bp5_operator_t op, const double *u_dev, double *out) {
  bp5_context_t ctx = op->ctx;
  const int n = op->n, n3 = n * n * n, nq = op->p + 2;
  const BlockGeom g = make_geom(op);
  L2Tables tb{};
  tb.nq = nq;
  double xq[kMaxN + 1], val[kMaxN], der[kMaxN];
  gauss_rule01(nq, xq, tb.w);
  for (int q = 0; q < nq; ++q) {
    lagrange_eval(n, op->tab.xi, xq[q], val, der);
    for (int i = 0; i < n; ++i) { tb.B[q * n + i] = val[i]; tb.D[q * n + i] = der[i]; }
  }
  // one CTA per cell; on a locally refined mesh per cell slot of the processing order (padding slots add zero)
  const long long n_blocks = op->hanging ? op->n_tiles * op->cells_per_tile : op->n_cells;
  L2Hanging hang{};
  BlockGeom gk = g;
  if (op->hanging) {
    hang.cells = static_cast<const int4 *>(op->hanging_cells);
    hang.tables = op->l2g_irr; hang.masks = op->cell_mask; hang.interp = op->hanging_interp_dev;
    for (int d = 0; d < 3; ++d) { gk.c0[d] = 0; hang.half[d] = 0.5 * g.h[d]; }
  }
  double *partial = nullptr;
  BP5_CUDA(cudaMalloc(&partial, sizeof(double) * (n_blocks + 1)));
  BP5_CUDA(cudaMemcpyToSymbolAsync(c_tab, &op->tab, sizeof(Tables1D), 0, cudaMemcpyHostToDevice, ctx->stream));
  const int threads = ((nq * nq * nq + 31) / 32) * 32;
  l2_norm_kernel<<<(unsigned)n_blocks, threads, sizeof(double) * (4 * n3 + 32), ctx->stream>>>(gk, tb, hang, u_dev, partial);
  BP5_CHECK_LAUNCH();
  sum_in_order_kernel<<<1, 256, 0, ctx->stream>>>(partial, n_blocks, partial + n_blocks);
  BP5_CHECK_LAUNCH();
  ctx->launches += 2;
  BP5_CUDA(cudaMemcpyAsync(out, partial + n_blocks, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  cudaFree(partial);
  return BP5_OK;
}

}  // namespace bp5
