// The BP5 hot kernel for sm_100a: what LocalPoissonOperator::operator()
// (bp5/step-64.cu:147-194) does through CUDAWrappers::FEEvaluation
// (read_dof_values / evaluate / merged coefficient / integrate /
// distribute_local_to_global; API mirrored by bp5/fe_evaluation_gl.h:133-250)
// inside MatrixFree::cell_loop's apply_kernel_shmem [UPSTREAM]; plus the
// Helmholtz variant of step-64/step-64.cu:201-219.
//
// Design (DESIGN.md section 3):
//  * persistent CTAs, a tile = CPT consecutive cells, tiles dealt round-robin so
//    that the set of cells in flight is one contiguous window of the mesh (L2
//    reuse of the gathered DoFs and of the dst lines being accumulated);
//  * the tile's metric ([cell][planes][n^3] fp64, 75-85 % of all bytes) is
//    fetched by ONE cp.async.bulk (TMA 1D) per tile into shared memory, signalled
//    on an mbarrier, and re-issued for the next tile as soon as the quadrature
//    phase has consumed it: tens of KB in flight per CTA with zero registers;
//  * DoF indices: one int per cell.  base >= 0: the cell's DoFs are affine in the
//    vector, idx(i,j,k) = base + i + j*sy + k*sz (structured numbering), so no
//    index stream is read at all; base < 0: explicit n^3-entry table (cells on a
//    partition's lower faces, whose ghost DoFs break the affine pattern).
//    Replaces the padded local_to_global array of bp5/fe_evaluation_gl.h:118,144.
//  * gathers for the next tile are issued into registers one tile ahead;
//  * contractions: n^2 threads per cell.  Each thread alternates between
//    "home" (owns the z-column (i,j,*)), "x-line" and "y-line" roles, holding a
//    whole line in registers, so one 1D contraction costs one shared-memory load
//    and one store per point instead of n loads; the z direction never leaves
//    registers.  Every contraction is done in even-odd form (EoShape below):
//    half the matrix operands and ~25-30 % fewer fp64 operations.  Shape matrices
//    are kernel parameters (constant bank), one private packed copy per direction,
//    so that ptxas has no cross-contraction reuse to cache in (and spill from) the
//    63 uniform registers (MOV.SPILL / R2UR.FILL per DFMA, measured 2x slower).
//  * scatter: DoFs interior to a cell have exactly one contribution: with
//    OVERWRITE they are written with a plain store (no zero-fill before, no
//    read-modify-write); only the skeleton (faces/edges/vertices) uses
//    fire-and-forget fp64 red.global.add into pre-zeroed entries.
#pragma once
#include <cuda_runtime.h>

#include <climits>
#include <cstdint>

#include "common.h"
#include "smem_layout.h"

namespace bp5 {

constexpr int kNoCell = INT_MIN;

// Shape tables as they travel to the kernel (by value, parameter constant bank).
// Even-odd form of a 1D matrix (deal.II's CPU evaluator uses the same decomposition [UPSTREAM
// evaluate_evenodd]): nodes and quadrature points are symmetric about the cell centre, so
// M[N-1-i][N-1-m] = S M[i][m] with S = +1 for values, -1 for derivatives (and their transposes).  With
// e[m] = v[m] + v[N-1-m], o[m] = v[m] - v[N-1-m] (m < H = N/2) only the first H1 = ceil(N/2) rows are needed:
//   pe = sum_m E[i][m] e[m] (+ C[i] v[H], N odd),  po = sum_m O[i][m] o[m],  out[i] = pe + po,  out[N-1-i] = S (pe - po)
// -- about N^2/2 + 2N fp64 operations and half the matrix operands instead of N^2.  Packed as E | O | C.
template <int N>
struct EoShape {
  static constexpr int H = N / 2, H1 = (N + 1) / 2;
  static constexpr int SIZE = 2 * H1 * H + H1;
};
// host: M is N x N row-major
template <int N>
inline void pack_matrix(double *dst, const double *M) {
  constexpr int H = EoShape<N>::H, H1 = EoShape<N>::H1;
  for (int i = 0; i < H1; ++i) {
    for (int m = 0; m < H; ++m) {
      dst[i * H + m] = 0.5 * (M[i * N + m] + M[i * N + (N - 1 - m)]);
      dst[H1 * H + i * H + m] = 0.5 * (M[i * N + m] - M[i * N + (N - 1 - m)]);
    }
    dst[2 * H1 * H + i] = (N % 2) ? M[i * N + H] : 0.0;
  }
}

template <int N>
struct KernelTables {
  // One private copy per coordinate direction (x, y, z): every unrolled contraction
  // then reads matrix entries nobody else reads, so ptxas has no cross-contraction
  // reuse to cache in (and spill from) the 63 uniform registers.
  double B[3][EoShape<N>::SIZE];     // B[q][i]: basis i at quadrature point q (identity for GLL)
  double BT[3][EoShape<N>::SIZE];    // transpose
  double D[3][EoShape<N>::SIZE];     // D[q][r]: derivative of the Lagrange basis through the QUADRATURE points
  double DT[3][EoShape<N>::SIZE];    // transpose
};
// host: fill all twelve copies from B[q][i] and D[q][r] (row-major N x N)
template <int N>
inline void fill_kernel_tables(KernelTables<N> &t, const double *B, const double *D) {
  double BT[N * N], DT[N * N];
  for (int q = 0; q < N; ++q)
    for (int i = 0; i < N; ++i) { BT[i * N + q] = B[q * N + i]; DT[i * N + q] = D[q * N + i]; }
  for (int d = 0; d < 3; ++d) {
    pack_matrix<N>(t.B[d], B); pack_matrix<N>(t.BT[d], BT);
    pack_matrix<N>(t.D[d], D); pack_matrix<N>(t.DT[d], DT);
  }
}

template <int N>
struct ApplyParams {
  const double *metric;   // [tile][CPT][PLANES][N^3], tile stride padded to 16 bytes
  const int *cell_base;   // [tiles*CPT]: >= 0 affine base, < 0: -(slot+1) into l2g_irr, kNoCell: padding
  const int *l2g_irr;     // [n_irregular][N^3] explicit local dof indices, x fastest
  const double *src;
  double *dst;
  long long tile_begin, n_tiles;   // tiles [tile_begin, n_tiles) of the processing order
  int sy, sz;             // affine strides of the owned box
  const int *skip;        // optional device flag: non-zero => nothing to do (CG already converged)
  double *dot_partials;   // OVERWRITE == 2: [gridDim.x] per-CTA parts of src . (A src), summed by the CG dots kernel
  KernelTables<N> tab;
  // AFFINE (geometry on the fly, affine mesh): G = w_q diag(aff) with aff = (hy hz / hx, hx hz / hy, hx hy / hz)
  // and the 1D quadrature weights wq.  (Behind `tab`: moving the tables in the parameter bank changes ptxas's
  // register allocation of the other kernels, p = 7 lost its third CTA per SM.)
  double aff[3];
  double wq[N];
  // HANG (locally refined mesh): constraint mask per cell slot and the two 1D parent-to-child interpolation matrices
  // [s][a * N + b] (operator_setup_hanging).  Appended for the same reason.
  const unsigned int *cell_mask;
  double hang[2][N * N];
  // cell_mask word, bits 8..10: stride class of an affine cell of a refined mesh (idx = base + i + j sy + k sz with
  // the class's strides: the numbering of a refined mesh is piecewise lexicographic)
  int hang_sy[8], hang_sz[8];
  // BLK (the merged CG's blocked layout, BlockedLayout in common.h): per-cell starts [4][blk_stride] in class A
  // (= cell_base), B, C and of the interior block; the offsets of a cell's upper y-face in class B and upper x-face in
  // class C; the non-face y planes (class C's run length) and the size of one z-face plane of class A
  const int *blk_desc;
  int blk_stride, blk_up_b, blk_up_c, blk_ji, blk_plane;
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!done);
}
// TMA 1D bulk copy global -> shared, completion on an mbarrier, L2 evict-first
// (the metric is streamed exactly once per operator application).
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar,
                                            uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t make_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

// 8-byte asynchronous copy global -> shared (LDGSTS): the one-tile-ahead gather without registers (kSmemPf)
__device__ __forceinline__ void cp_async8(void *smem_dst, const void *gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Local dof indices of the N points of one thread's z-column in a cell with
// descriptor `base` (>= 0: affine, < 0: explicit table slot, kNoCell: no cell,
// indices are 0 and the values are never used).  Branch-free on the common path
// so that the N value loads that follow are issued back to back.
template <int N>
__device__ __forceinline__ void column_indices(int (&idx)[N], const int *__restrict__ l2g_irr, int base, int ab_off,
                                               int ab_irr, int sz) {
  if (base >= 0 || base == kNoCell) {
    const int b0 = base >= 0 ? base + ab_off : 0;
    const int s = base >= 0 ? sz : 0;
#pragma unroll
    for (int k = 0; k < N; ++k) idx[k] = b0 + k * s;
  } else {
    const int *row = l2g_irr + (long long)(-(base + 1)) * (N * N * N) + ab_irr;
#pragma unroll
    for (int k = 0; k < N; ++k) idx[k] = __ldg(row + k * N * N);
  }
}

// The same in the blocked layout: the column's ends lie on the cell's two z-faces (class A, one plane apart), the points
// between them in one run of class B, C or the interior block (m0 + k m_str, m_off and m_str per thread).
template <int N>
__device__ __forceinline__ void column_indices_blk(int (&idx)[N], int base, int ab_off, int mbase, int m_off,
                                                   int m_str, int plane) {
  const bool cell = base != kNoCell;
  const int a0 = cell ? base + ab_off : 0, m0 = cell ? mbase + m_off : 0, s = cell ? m_str : 0;
  idx[0] = a0;
  idx[N - 1] = cell ? a0 + plane : 0;
#pragma unroll
  for (int k = 1; k < N - 1; ++k) idx[k] = m0 + k * s;
}

// w = M v for a matrix with symmetry sign S (see EoShape); fully unrolled, result in registers (indexed statically)
template <int N, int S>
__device__ __forceinline__ void contract_in_regs(double (&w)[N], const double *__restrict__ M, const double (&v)[N]) {
  constexpr int H = EoShape<N>::H, H1 = EoShape<N>::H1;
  const double *__restrict__ E = M, *__restrict__ O = M + H1 * H, *__restrict__ C = M + 2 * H1 * H;
  double e[H > 0 ? H : 1], o[H > 0 ? H : 1];
#pragma unroll
  for (int m = 0; m < H; ++m) { e[m] = v[m] + v[N - 1 - m]; o[m] = v[m] - v[N - 1 - m]; }
#pragma unroll
  for (int i = 0; i < H; ++i) {
    double pe = (N % 2) ? C[i] * v[H] : 0.0, po = 0.0;
#pragma unroll
    for (int m = 0; m < H; ++m) { pe += E[i * H + m] * e[m]; po += O[i * H + m] * o[m]; }
    w[i] = pe + po;
    w[N - 1 - i] = S > 0 ? pe - po : po - pe;
  }
  if (N % 2) {
    double mid = S > 0 ? C[H] * v[H] : 0.0;
#pragma unroll
    for (int m = 0; m < H; ++m) mid += (S > 0 ? E[H * H + m] * e[m] : O[H * H + m] * o[m]);
    w[H] = mid;
  }
}

// out[i*stride] = sum_m M[i][m] v[m]
template <int N, int S>
__device__ __forceinline__ void contract_to_smem(double *out, int stride, const double *__restrict__ M,
                                                 const double (&v)[N]) {
  double w[N];
  contract_in_regs<N, S>(w, M, v);
#pragma unroll
  for (int i = 0; i < N; ++i) out[i * stride] = w[i];
}

// ---- hanging-node constraints of the children of a locally refined mesh (HANG kernels only) ----------------------
// A node on a constrained face was gathered from the unrefined neighbour's face DoF of the same local index; the
// child's values are the neighbour's face polynomial at the child's nodes: 1D interpolations along the face's two
// tangential directions (bp5/fe_evaluation_gl.h:150,167, resolve_hanging_nodes).  mask: bit d = face normal to d
// constrained, bit 3+d = position of the child in its parent (face at node 0 or p; which matrix).
// Direction by direction every line inside a constrained face is interpolated once; z-lines are the home columns
// (registers), x- and y-lines go through the layout-A array `arr` like the contractions.  T: the transposes, for the
// scatter.  Called by ALL threads of a CTA whose tile has a masked cell (barriers inside).
template <int N, bool T>
__device__ __forceinline__ void hang_matvec(double (&v)[N], const double *__restrict__ M) {
  double w[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
    double sum = 0.0;
#pragma unroll
    for (int m = 0; m < N; ++m) sum += (T ? M[m * N + i] : M[i * N + m]) * v[m];
    w[i] = sum;
  }
#pragma unroll
  for (int i = 0; i < N; ++i) v[i] = w[i];
}

// The home columns are exchanged through `arr` by the caller (publish before, reload after), so that no register array
// crosses this (deliberately not inlined) function: the main loop keeps its register allocation and has no stack.
template <int N, bool T, int A1, int A2>
__device__ __noinline__ void hang_exchange(unsigned int mask, bool active, int a, int b, double *arr,
                                           const double (*hang)[N * N]) {
  const int hA = b * A1 + a, xA = b * A2 + a * A1, yA = b * A2 + a;
  const int f0 = ((mask >> 3) & 1u) ? N - 1 : 0, f1 = ((mask >> 4) & 1u) ? N - 1 : 0, f2 = ((mask >> 5) & 1u) ? N - 1 : 0;
  const bool c0 = (mask & 1u) != 0, c1 = (mask & 2u) != 0, c2 = (mask & 4u) != 0;
  const double *M0 = hang[(mask >> 3) & 1u], *M1 = hang[(mask >> 4) & 1u], *M2 = hang[(mask >> 5) & 1u];
  // home column (i=a, j=b): a z-line; it lies in the constrained x-face if a == f0, in the y-face if b == f1
  const bool z_line = active && ((c0 && a == f0) || (c1 && b == f1));
  // x-line role (j=a, k=b): in the y-face if a == f1, in the z-face if b == f2
  const bool x_line = active && ((c1 && a == f1) || (c2 && b == f2));
  // y-line role (i=a, k=b): in the x-face if a == f0, in the z-face if b == f2
  const bool y_line = active && ((c0 && a == f0) || (c2 && b == f2));
  auto line = [&](int at, int st, const double *M) {
    double v[N];
#pragma unroll
    for (int m = 0; m < N; ++m) v[m] = arr[at + m * st];
    hang_matvec<N, T>(v, M);
#pragma unroll
    for (int m = 0; m < N; ++m) arr[at + m * st] = v[m];
  };
  // forward: z (own column, just published by this thread), x, y; transpose: y, x, z
  if (!T && z_line) line(hA, A2, M2);
  __syncthreads();
  if (T ? y_line : x_line) line(T ? yA : xA, T ? A1 : 1, T ? M1 : M0);
  __syncthreads();
  if (T ? x_line : y_line) line(T ? xA : yA, T ? 1 : A1, T ? M0 : M1);
  __syncthreads();
  if (T && z_line) line(hA, A2, M2);
}

// AFFINE: where G comes from.
//   false: the stored metric, one TMA bulk copy per tile into shared memory (mbarrier), read back with LDS
//          (measured faster than streaming it into registers, profiles/r1_v3_notes.md section 3);
//   true:  no metric at all -- geometry on the fly on an AFFINE (axis-parallel) mesh: the Jacobian is one constant
//          diagonal, G = w_q diag(hy hz / hx, hx hz / hy, hx hy / hz) is formed from kernel parameters.
//          16 bytes per DoF of HBM traffic instead of 16 + 48 r: shared-memory-pipe / fp64 bound.
// The kernels leave the minimum of resident CTAs per SM to ptxas's heuristic: an explicit minimum of 1 makes it spend
// ~50 more registers.
template <int P, int CPT, int PLANES, bool AFFINE = false>
struct ApplyCfg {
  static constexpr int N = P + 1, N2 = N * N, N3 = N2 * N;
  using L = SmemLayout<N, CPT>;                            // per-array bank-conflict-minimising strides
  static constexpr int ACTIVE = CPT * N2;
  static constexpr int NT = ((ACTIVE + 31) / 32) * 32;
  static constexpr int METRIC_DOUBLES = (CPT * PLANES * N3 + 1) & ~1;  // per tile, padded to 16 bytes
  static constexpr uint32_t METRIC_BYTES = METRIC_DOUBLES * 8;
  static constexpr int WORK_DOUBLES = CPT * (2 * L::A_CS + L::B_CS);   // S0, S1 (layout A) and S2 (layout B)
  static constexpr int STAGE_DOUBLES = AFFINE ? 0 : METRIC_DOUBLES;   // shared-memory staging of the metric
  // the mbarrier (8 bytes) goes into the padding word at the end of the first cell's S0 array when the layout
  // leaves one free, else behind the work arrays: at p = 7 those 16 bytes decide between 2 and 3 CTAs per SM
  // (3 x (76800 + 1024 reserved) = 233472 bytes = all of an SM's shared memory)
  static constexpr int A_LAST = (N - 1) * (L::A_S2 + L::A_S1 + 1);           // last used index of a layout-A array
  static constexpr bool BAR_IN_PAD = L::A_CS - 1 > A_LAST;
  static constexpr size_t SMEM_BYTES = (size_t)STAGE_DOUBLES * 8 + (size_t)WORK_DOUBLES * 8 + (BAR_IN_PAD ? 0 : 16);
  static_assert(!AFFINE || PLANES == 6, "the affine fast path is for the Poisson operator");
  static_assert(METRIC_BYTES % 16 == 0, "bulk copy size must be a multiple of 16 bytes");
};

// QUAD: 0 = Gauss (basis nodes != quadrature points: interpolate, then
// collocation derivative), 1 = Gauss-Lobatto collocation (B = identity).
// HELM: 0 = Poisson (6 planes), 1 = Helmholtz (7th plane a(x) JxW on the values).
// OVERWRITE: 2 = like 1, and the CTA also reduces src . (A src) over its cells, evaluated at the
// quadrature points as sum_q g_q^T G_q g_q (+ mass term) -- the "p.v" dot product of the merged CG
// (bp5/solver.h:231,303) without reading either vector again;
// 1 = cell-interior DoFs are stored, not added (dst's skeleton must be
// zero on entry, its interior may hold anything); 0 = dst += A src everywhere.
// OVERWRITE + 3 (3, 4, 5): the same with plain read-modify-writes in place of the atomics, for the launches over
// the tiles of ONE colour of the coloured cell order (cells of a colour share no DoF): bitwise reproducible.
// HANG (locally refined meshes): 1 = the cells may carry hanging-node constraints (prm.cell_mask), resolved after the
// gather and before the scatter -- one extra CTA-wide vote per tile, the exchange passes only in tiles that hold a masked
// cell; 2 = no constrained cell in the tile range, only the per-cell stride classes of the refined numbering.
// BLK: src and dst in the merged CG's blocked layout (conforming single block, default cell order); cell_base holds the
// cells' class-A starts and prm.blk_desc the others.  Interior DoFs then share no sector with the skeleton.
template <int P, int QUAD, int HELM, int CPT, int OWMODE, bool AFFINE = false, int HANG = 0, bool BLK = false>
__device__ __forceinline__ void bp5_apply_body(const ApplyParams<P + 1> &prm) {
  static_assert(!BLK || (HANG == 0 && OWMODE < 3), "the blocked layout is for the conforming, uncoloured kernels");
  constexpr int OVERWRITE = OWMODE % 3;
  constexpr bool PLAIN_ADD = OWMODE >= 3;
  using Cfg = ApplyCfg<P, CPT, 6 + HELM, AFFINE>;
  constexpr int N = Cfg::N, N2 = Cfg::N2, N3 = Cfg::N3, PLANES = 6 + HELM;
  using L = typename Cfg::L;
  constexpr int A1 = L::A_S1, A2 = L::A_S2, B1 = L::B_S1, B2 = L::B_S2;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double *Gs = reinterpret_cast<double *>(smem_raw);                 // [CPT][PLANES][N3]
  double *S0 = Gs + Cfg::STAGE_DOUBLES;                              // layout A (home + x-line + y-line readers)
  double *S1 = S0 + CPT * L::A_CS;                                   // layout A (home + x-line)
  double *S2 = S1 + CPT * L::A_CS;                                   // layout B (home + y-line)
  uint64_t *bar = reinterpret_cast<uint64_t *>(Cfg::BAR_IN_PAD ? S0 + L::A_CS - 1 : S2 + CPT * L::B_CS);

  if (prm.skip != nullptr && *prm.skip != 0) return;
  const int tid = threadIdx.x;
  const bool active = tid < Cfg::ACTIVE;
  const int c = active ? tid / N2 : 0;      // cell within the tile
  const int r = tid % N2;
  const int a = r % N, b = r / N;           // the two free indices of this thread's line/column
  double *s0 = S0 + c * L::A_CS, *s1 = S1 + c * L::A_CS, *s2 = S2 + c * L::B_CS;
  const double *gm = Gs + c * PLANES * N3;
  const double *__restrict__ Bx = prm.tab.B[0], *__restrict__ By = prm.tab.B[1], *__restrict__ Bz = prm.tab.B[2];
  const double *__restrict__ BTx = prm.tab.BT[0], *__restrict__ BTy = prm.tab.BT[1], *__restrict__ BTz = prm.tab.BT[2];
  const double *__restrict__ Dx = prm.tab.D[0], *__restrict__ Dy = prm.tab.D[1], *__restrict__ Dz = prm.tab.D[2];
  const double *__restrict__ DTx = prm.tab.DT[0], *__restrict__ DTy = prm.tab.DT[1], *__restrict__ DTz = prm.tab.DT[2];
  const int ab_off = a + b * prm.sy;        // affine offset of this thread's column
  const int ab_irr = b * N + a;
  // shared-memory offsets of this thread's three roles
  // address(i,j,k) = k*S2 + j*S1 + i in each array's own strides
  const int hA = b * A1 + a, hB = b * B1 + a;     // + k * {A2,B2} : home column (i=a, j=b, k)
  const int xA = b * A2 + a * A1;                 // + i           : x-line (i, j=a, k=b)
  const int yA = b * A2 + a, yB = b * B2 + a;     // + j * {A1,B1} : y-line (i=a, j, k=b)

  const long long tile0 = prm.tile_begin + blockIdx.x;
  const long long tstride = gridDim.x;
  const long long n_tiles = prm.n_tiles;
  const int sz = prm.sz;
  const int *__restrict__ cell_base = prm.cell_base;
  const int *__restrict__ l2g_irr = prm.l2g_irr;
  const double *__restrict__ src = prm.src;
  double *__restrict__ dst = prm.dst;
  // prm.metric is read where the TMA copies are issued: a local copy of it is loaded once at the top of the kernel,
  // and that changes ptxas's register allocation of the stored-metric kernels at most degrees
  uint64_t policy = 0;
  if constexpr (!AFFINE) {
    if (tid == 0) {
      mbar_init(bar, 1);
      fence_barrier_init();
      policy = make_evict_first_policy();
      if (tile0 < n_tiles) {
        mbar_expect_tx(bar, Cfg::METRIC_BYTES);
        tma_load_1d(Gs, prm.metric + tile0 * (long long)Cfg::METRIC_DOUBLES, Cfg::METRIC_BYTES, bar, policy);
      }
    }
    __syncthreads();
  }
  [[maybe_unused]] const double wab = AFFINE ? prm.wq[a] * prm.wq[b] : 0.0;

  // software pipeline of the gather: cell descriptors two tiles ahead, values one tile ahead
  int base_cur = (active && tile0 < n_tiles) ? __ldg(cell_base + tile0 * CPT + c) : kNoCell;
  int base_nxt = (active && tile0 + tstride < n_tiles) ? __ldg(cell_base + (tile0 + tstride) * CPT + c) : kNoCell;
  // kSmemPf (p = 8 collocation, conforming meshes): the next tile's columns are copied asynchronously (LDGSTS)
  // straight into S0 -- free from the end of the line phase (2) to the next tile's start -- instead of waiting in N
  // registers: the copy replaces the publishing stores, the home thread reads its column back for the z-derivative.
  // ptxas then needs 48-78 instead of 106-194 registers.  Measured at 148 M DoFs (profiles/r2_smem_prefetch_probe.log):
  // p = 8 cell loop 2.67 -> 2.33 ms (2 -> 4 CTAs/SM), merged CG 32.8 -> 34.8 GDoF*it/s; p = 5, 6 (shared memory
  // already limits the CTAs) 1-2 % slower -- the copy is in flight for 60 % of a tile instead of a whole one.
  // Everywhere else the values of the next tile wait in registers (kPrefetch): without that prefetch p = 5, 6 gain a
  // CTA per SM and still lose 9-13 % of the CG rate (profiles/r2_no_prefetch_p56_probe.log).
  constexpr bool kSmemPf = P == 8 && QUAD == 1 && HANG == 0;
  constexpr bool kPrefetch = !kSmemPf;   // values of the next tile in registers one tile ahead
  // HANG: the mask words travel with the cell descriptors (they select the strides of the gather)
  [[maybe_unused]] unsigned int w_cur = 0, w_nxt = 0;
  if constexpr (HANG) {
    w_cur = (active && tile0 < n_tiles) ? __ldg(prm.cell_mask + tile0 * CPT + c) : 0u;
    w_nxt = (active && tile0 + tstride < n_tiles) ? __ldg(prm.cell_mask + (tile0 + tstride) * CPT + c) : 0u;
  }
  auto off_of = [&](unsigned int w) { return HANG ? a + b * prm.hang_sy[(w >> 8) & 7u] : ab_off; };
  auto sz_of = [&](unsigned int w) { return HANG ? prm.hang_sz[(w >> 8) & 7u] : sz; };
  // BLK: the class of this thread's column between the z-faces (1: B, on a y-face; 2: C, on an x-face only; 3: interior
  // block), its offset in the cell's run and its stride; the cells' starts in that class travel with the descriptors
  [[maybe_unused]] int m_cls = 0, m_off = 0, m_str = 0, m_cur = 0, m_nxt = 0;
  if constexpr (BLK) {
    const bool yface = b == 0 || b == P, xface = a == 0 || a == P;
    m_cls = yface ? 1 : xface ? 2 : 3;
    m_str = yface ? prm.sy : xface ? prm.blk_ji : (P - 1) * (P - 1);
    m_off = (yface ? a + (b == P ? prm.blk_up_b : 0) : xface ? b - 1 + (a == P ? prm.blk_up_c : 0) : (b - 1) * (P - 1) + a - 1) -
            m_str;
    m_cur = (active && tile0 < n_tiles) ? __ldg(prm.blk_desc + m_cls * prm.blk_stride + tile0 * CPT + c) : 0;
    m_nxt = (active && tile0 + tstride < n_tiles) ? __ldg(prm.blk_desc + m_cls * prm.blk_stride + (tile0 + tstride) * CPT + c)
                                                  : 0;
  }
  auto indices = [&](int (&idx)[N], int base, unsigned int w, int mbase) {
    if constexpr (BLK) column_indices_blk<N>(idx, base, ab_off, mbase, m_off, m_str, prm.blk_plane);
    else column_indices<N>(idx, l2g_irr, base, off_of(w), ab_irr, sz_of(w));
  };
  auto gather = [&](double (&u)[N], int base, unsigned int w, int mbase) {
    int idx[N];
    indices(idx, base, w, mbase);
#pragma unroll
    for (int k = 0; k < N; ++k) u[k] = __ldg(src + idx[k]);
  };
  [[maybe_unused]] double u_nxt[N];
  if constexpr (kPrefetch) gather(u_nxt, base_cur, w_cur, m_cur);
  if constexpr (kSmemPf) {
    if (active && tile0 < n_tiles) {
      int ix[N];
      indices(ix, base_cur, w_cur, m_cur);
#pragma unroll
      for (int k = 0; k < N; ++k) cp_async8(s0 + hA + k * A2, src + ix[k]);
    }
  }

  uint32_t parity = 0;
  [[maybe_unused]] double dot_acc = 0.0;
  for (long long tile = tile0; tile < n_tiles; tile += tstride) {
    double u[N];
#pragma unroll
    for (int k = 0; k < N; ++k) u[k] = kPrefetch ? u_nxt[k] : 0.0;
    if constexpr (kSmemPf) {
      cp_async_wait_all();      // this thread's own column has landed (the others': behind the barrier of phase 1)
      if (active) {
#pragma unroll
        for (int k = 0; k < N; ++k) u[k] = s0[hA + k * A2];
      }
    } else if constexpr (!kPrefetch) gather(u, base_cur, w_cur, m_cur);
    // issue next tile's gather and the descriptor load of the tile after it
    if constexpr (kPrefetch) gather(u_nxt, base_nxt, w_nxt, m_nxt);
    const int base_n2 =
        (active && tile + 2 * tstride < n_tiles) ? __ldg(cell_base + (tile + 2 * tstride) * CPT + c) : kNoCell;
    [[maybe_unused]] unsigned int w_n2 = 0;
    if constexpr (HANG)
      w_n2 = (active && tile + 2 * tstride < n_tiles) ? __ldg(prm.cell_mask + (tile + 2 * tstride) * CPT + c) : 0u;
    [[maybe_unused]] int m_n2 = 0;
    if constexpr (BLK)
      m_n2 = (active && tile + 2 * tstride < n_tiles)
                 ? __ldg(prm.blk_desc + m_cls * prm.blk_stride + (tile + 2 * tstride) * CPT + c)
                 : 0;

    [[maybe_unused]] unsigned int hmask = 0;
    [[maybe_unused]] bool tile_hangs = false;
    if constexpr (HANG == 1) {
      hmask = w_cur & 63u;
      tile_hangs = __syncthreads_or(hmask != 0) != 0;
      if (tile_hangs) {
        if (active) {
#pragma unroll
          for (int k = 0; k < N; ++k) s0[hA + k * A2] = u[k];
        }
        hang_exchange<N, false, A1, A2>(hmask, active, a, b, s0, prm.hang);
        if (active && hmask != 0) {
#pragma unroll
          for (int k = 0; k < N; ++k) u[k] = s0[hA + k * A2];
        }
      }
    }
    double t[N];   // z-direction data that stays in registers across the quadrature phase
    double mv[N];  // Helmholtz: values at the quadrature points (home column)

    if constexpr (QUAD == 1) {
      // ---------------- Gauss-Lobatto collocation: u is already at the q-points
      // (1) home (i=a, j=b): publish the column, z-derivative in registers
      if (active) {
        if constexpr (!kSmemPf) {
#pragma unroll
          for (int k = 0; k < N; ++k) s0[hA + k * A2] = u[k];
        }
        contract_in_regs<N, -1>(t, Dz, u);
        if constexpr (HELM) {
#pragma unroll
          for (int k = 0; k < N; ++k) mv[k] = u[k];
        }
      }
      __syncthreads();
      // (2) x-line (j=a, k=b) and y-line (i=a, k=b): derivative along the line
      if (active) {
        double v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = s0[xA + i];
        contract_to_smem<N, -1>(s1 + xA, 1, Dx, v);
#pragma unroll
        for (int j = 0; j < N; ++j) v[j] = s0[yA + j * A1];
        contract_to_smem<N, -1>(s2 + yB, B1, Dy, v);
      }
      __syncthreads();
      if constexpr (kSmemPf) {   // S0 is free until the next tile starts: fetch its columns behind the rest of this one
        if (active && tile + tstride < n_tiles) {
          int ix[N];
          indices(ix, base_nxt, w_nxt, m_nxt);
#pragma unroll
          for (int k = 0; k < N; ++k) cp_async8(s0 + hA + k * A2, src + ix[k]);
        }
      }
    } else {
      // ---------------- Gauss quadrature: interpolate to the q-points first
      // (1) home (i=a, j=b): z-interpolation
      if (active) contract_to_smem<N, 1>(s0 + hA, A2, Bz, u);
      __syncthreads();
      // (2) x-line (j=a, qz=b): x-interpolation in place
      if (active) {
        double v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = s0[xA + i];
        contract_to_smem<N, 1>(s0 + xA, 1, Bx, v);
      }
      __syncthreads();
      // (3) y-line (qx=a, qz=b): y-interpolation (values at q-points), then d/dy
      if (active) {
        double v[N], w[N];
#pragma unroll
        for (int j = 0; j < N; ++j) v[j] = s0[yA + j * A1];
        contract_in_regs<N, 1>(w, By, v);
#pragma unroll
        for (int q = 0; q < N; ++q) s0[yA + q * A1] = w[q];
        contract_to_smem<N, -1>(s2 + yB, B1, Dy, w);
      }
      __syncthreads();
      // (4) x-line (qy=a, qz=b): d/dx ; home (qx=a, qy=b): d/dz in registers
      if (active) {
        double v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = s0[xA + i];
        contract_to_smem<N, -1>(s1 + xA, 1, Dx, v);
#pragma unroll
        for (int k = 0; k < N; ++k) v[k] = s0[hA + k * A2];
        contract_in_regs<N, -1>(t, Dz, v);
        if constexpr (HELM) {
#pragma unroll
          for (int k = 0; k < N; ++k) mv[k] = v[k];
        }
      }
      __syncthreads();
    }

    // ---------------- quadrature-point phase (home): g <- G g  (bp5/step-64.cu:160-188)
    if constexpr (!AFFINE) {
      mbar_wait(bar, parity);
      parity ^= 1;
    }
    if (active) {
#pragma unroll
      for (int k = 0; k < N; ++k) {
        const int q = (k * N + b) * N + a, wA = hA + k * A2, wB = hB + k * B2;
        const double ur = s1[wA], us = s2[wB], ut = t[k];
        double g0, g1, g2, g3, g4, g5;
        if constexpr (AFFINE) {
          const double w = wab * prm.wq[k];
          g0 = prm.aff[0] * w; g1 = prm.aff[1] * w; g2 = prm.aff[2] * w; g3 = g4 = g5 = 0.0;
        } else {
          g0 = gm[q]; g1 = gm[N3 + q]; g2 = gm[2 * N3 + q]; g3 = gm[3 * N3 + q]; g4 = gm[4 * N3 + q]; g5 = gm[5 * N3 + q];
        }
        const double vr = ur * g0 + us * g3 + ut * g4;
        const double vs = ur * g3 + us * g1 + ut * g5;
        const double vt = ur * g4 + us * g5 + ut * g2;
        s1[wA] = vr;
        s2[wB] = vs;
        t[k] = vt;
        if constexpr (OVERWRITE == 2) dot_acc += ur * vr + us * vs + ut * vt;
        if constexpr (HELM) {
          const double m_old = mv[k];
          mv[k] = m_old * gm[6 * N3 + q];
          if constexpr (OVERWRITE == 2) dot_acc += m_old * mv[k];
        }
      }
    }
    __syncthreads();
    if constexpr (!AFFINE) {
      // the metric buffer is free: fetch the next tile's metric behind the remaining work
      if (tid == 0 && tile + tstride < n_tiles) {
        mbar_expect_tx(bar, Cfg::METRIC_BYTES);
        tma_load_1d(Gs, prm.metric + (tile + tstride) * (long long)Cfg::METRIC_DOUBLES, Cfg::METRIC_BYTES, bar, policy);
      }
    }

    int idx[N];
    indices(idx, base_cur, w_cur, m_cur);
    const bool col_interior = OVERWRITE != 0 && a > 0 && a < P && b > 0 && b < P;
    const bool do_scatter = base_cur != kNoCell;

    if constexpr (QUAD == 1) {
      // (4) transposed derivative along x- and y-lines, in place
      if (active) {
        double v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = s1[xA + i];
        contract_to_smem<N, -1>(s1 + xA, 1, DTx, v);
#pragma unroll
        for (int j = 0; j < N; ++j) v[j] = s2[yB + j * B1];
        contract_to_smem<N, -1>(s2 + yB, B1, DTy, v);
      }
      __syncthreads();
      // (5) home: z-transpose in registers, sum the three directions, scatter
      if constexpr (HANG != 1) {
        if (do_scatter) {
          double o[N];
          contract_in_regs<N, -1>(o, DTz, t);
#pragma unroll
          for (int k = 0; k < N; ++k) {
            double s = o[k] + s1[hA + k * A2] + s2[hB + k * B2];
            if constexpr (HELM) s += mv[k];
            double *dp = dst + idx[k];
            if (col_interior && k > 0 && k < P) *dp = s;     // multiplicity 1: plain store
            else if constexpr (PLAIN_ADD) *dp += s;          // one colour per launch: no other cell touches this DoF
            else atomicAdd(dp, s);                           // skeleton: red.global.add.f64
          }
        }
      } else {
        double o[N];
        if (do_scatter) {
          contract_in_regs<N, -1>(o, DTz, t);
#pragma unroll
          for (int k = 0; k < N; ++k) {
            o[k] += s1[hA + k * A2] + s2[hB + k * B2];
            if constexpr (HELM) o[k] += mv[k];
          }
        }
        if (tile_hangs) {   // s0 is free since (2)
          if (active) {
#pragma unroll
            for (int k = 0; k < N; ++k) s0[hA + k * A2] = o[k];
          }
          hang_exchange<N, true, A1, A2>(hmask, active, a, b, s0, prm.hang);
          if (active && hmask != 0) {
#pragma unroll
            for (int k = 0; k < N; ++k) o[k] = s0[hA + k * A2];
          }
        }
        if (do_scatter) {
#pragma unroll
          for (int k = 0; k < N; ++k) {
            double *dp = dst + idx[k];
            if (col_interior && k > 0 && k < P) *dp = o[k];
            else atomicAdd(dp, o[k]);
          }
        }
      }
    } else {
      // (6a) x-line: D^T along x in place ; home: D^T along z (+ mass term) -> S0
      if (active) {
        double v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = s1[xA + i];
        contract_to_smem<N, -1>(s1 + xA, 1, DTx, v);
        if constexpr (HELM) {
          double o[N];
          contract_in_regs<N, -1>(o, DTz, t);
#pragma unroll
          for (int k = 0; k < N; ++k) s0[hA + k * A2] = o[k] + mv[k];
        } else {
          contract_to_smem<N, -1>(s0 + hA, A2, DTz, t);
        }
      }
      __syncthreads();
      // (6b) y-line (qx=a, qz=b): D^T along y, add x and z parts, then B^T along y
      if (active) {
        double v[N], y[N];
#pragma unroll
        for (int q = 0; q < N; ++q) v[q] = s2[yB + q * B1];
        contract_in_regs<N, -1>(y, DTy, v);
#pragma unroll
        for (int q = 0; q < N; ++q) y[q] += s1[yA + q * A1] + s0[yA + q * A1];
        contract_to_smem<N, 1>(s0 + yA, A1, BTy, y);
      }
      __syncthreads();
      // (7) x-line (j=a, qz=b): B^T along x in place
      if (active) {
        double v[N];
#pragma unroll
        for (int q = 0; q < N; ++q) v[q] = s0[xA + q];
        contract_to_smem<N, 1>(s0 + xA, 1, BTx, v);
      }
      __syncthreads();
      // (8) home (i=a, j=b): B^T along z in registers, scatter
      if constexpr (HANG != 1) {
        if (do_scatter) {
          double v[N], o[N];
#pragma unroll
          for (int q = 0; q < N; ++q) v[q] = s0[hA + q * A2];
          contract_in_regs<N, 1>(o, BTz, v);
#pragma unroll
          for (int k = 0; k < N; ++k) {
            double *dp = dst + idx[k];
            if (col_interior && k > 0 && k < P) *dp = o[k];
            else if constexpr (PLAIN_ADD) *dp += o[k];
            else atomicAdd(dp, o[k]);
          }
        }
      } else {
        double o[N];
        if (do_scatter) {
          double v[N];
#pragma unroll
          for (int q = 0; q < N; ++q) v[q] = s0[hA + q * A2];
          contract_in_regs<N, 1>(o, BTz, v);
        }
        if (tile_hangs) {   // s1 is free since (6b)
          if (active) {
#pragma unroll
            for (int k = 0; k < N; ++k) s1[hA + k * A2] = o[k];
          }
          hang_exchange<N, true, A1, A2>(hmask, active, a, b, s1, prm.hang);
          if (active && hmask != 0) {
#pragma unroll
            for (int k = 0; k < N; ++k) o[k] = s1[hA + k * A2];
          }
        }
        if (do_scatter) {
#pragma unroll
          for (int k = 0; k < N; ++k) {
            double *dp = dst + idx[k];
            if (col_interior && k > 0 && k < P) *dp = o[k];
            else atomicAdd(dp, o[k]);
          }
        }
      }
    }
    base_cur = base_nxt;
    base_nxt = base_n2;
    if constexpr (HANG) { w_cur = w_nxt; w_nxt = w_n2; }
    if constexpr (BLK) { m_cur = m_nxt; m_nxt = m_n2; }
  }
  if constexpr (OVERWRITE == 2) {
    // CTA-wide sum in a fixed order (warp shuffles, then warp 0 over the per-warp sums)
    __syncthreads();
    double v = active ? dot_acc : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((tid & 31) == 0) S0[tid >> 5] = v;
    __syncthreads();
    if (tid < 32) {
      v = tid < Cfg::NT / 32 ? S0[tid] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (tid == 0) prm.dot_partials[blockIdx.x] = v;
    }
  }
}

template <int P, int QUAD, int HELM, int CPT, int OWMODE, bool AFFINE = false, bool BLK = false>
__global__ void __launch_bounds__(ApplyCfg<P, CPT, 6 + HELM, AFFINE>::NT)
    bp5_apply_kernel(const __grid_constant__ ApplyParams<P + 1> prm) {
  bp5_apply_body<P, QUAD, HELM, CPT, OWMODE, AFFINE, 0, BLK>(prm);
}

// The kernels for locally refined meshes.  Their main loop is the conforming kernel's; the (not inlined) constraint
// exchange would raise the kernel's register count to 200+ and halve the resident CTAs, so the register budget of the
// conforming kernel is imposed (the exchange spills inside its own frame, in the few tiles that hold a masked cell):
// <= 128 registers up to p = 6 (16 warps/SM), 168 at p = 7, 8 (12 warps).  Measured on a half-refined corner
// (profiles/r2_refined_mesh_probe.jsonl), vmult GDoF/s p = 4 / 6 / 7 / 8: exchange inlined, no budget (192-226 registers)
// 30.4 / 25.3 / - / 22.6; this arrangement 30.3 / 34.6 / 37.6 / 32.4 (p = 8: budget 168); a 168 budget for all degrees
// through -maxrregcount without launch bounds 27.2 / 25.1 / 32.6 / 32.4.
template <int P, int NT>
constexpr int hang_min_blocks() {
  constexpr int warps = (NT + 31) / 32;
  return (P <= 6 ? 16 : 12) / warps;
}
template <int P, int QUAD, int HELM, int CPT, int OWMODE>
__global__ void __launch_bounds__((ApplyCfg<P, CPT, 6 + HELM>::NT), (hang_min_blocks<P, ApplyCfg<P, CPT, 6 + HELM>::NT>()))
    bp5_apply_hang_kernel(const __grid_constant__ ApplyParams<P + 1> prm) {
  bp5_apply_body<P, QUAD, HELM, CPT, OWMODE, false, 1>(prm);
}
// the affine cells of a refined mesh: the conforming kernel plus the stride class per cell
template <int P, int QUAD, int HELM, int CPT, int OWMODE>
__global__ void __launch_bounds__(ApplyCfg<P, CPT, 6 + HELM>::NT)
    bp5_apply_strided_kernel(const __grid_constant__ ApplyParams<P + 1> prm) {
  bp5_apply_body<P, QUAD, HELM, CPT, OWMODE, false, 2>(prm);
}

}  // namespace bp5
