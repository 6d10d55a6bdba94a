// BP5 cell kernel with ON-THE-FLY geometry (BASELINE config 5, "stored metric tensor vs on-the-fly
// geometry"): instead of streaming the merged coefficient G = JxW J^-1 J^-T (48 bytes per quadrature
// point, what evaluate_coefficients(JacobianFunctor) precomputes, bp5/step-64.cu:84-114,256-258) the
// kernel gathers the nodal coordinates of the degree-p mapped cell (24 bytes per DoF, the support points
// MappingQGeneric(p) interpolates, bp5/step-64.cu:234), differentiates them with the same collocation
// sum factorisation as the solution (nine more 1D contractions) and forms G at every point:
//     J[d][e] = d x_d / d xi_e,   G = w_q / det(J) * adj(J) adj(J)^T   (== JxW J^-1 J^-T).
// Gauss-Lobatto collocation only (nodes == quadrature points).  Same tiles, thread roles, shared-memory
// layouts, scatter and fused d.(A d) as apply.cuh; no TMA stage (there is no metric stream).
// Algorithmic bytes: 16 (src, dst) + 24 (coordinates) per DoF instead of 16 + 48 ((p+1)/p)^3.
#pragma once
#include "apply.cuh"

namespace bp5 {

template <int N>
struct ApplyOtfParams {
  const double *cx, *cy, *cz;   // nodal coordinates per local DoF (owned, then ghost), same indexing as src
  const int *cell_base;
  const int *l2g_irr;
  const double *src;
  double *dst;
  long long tile_begin, n_tiles;
  int sy, sz;
  const int *skip;
  double *dot_partials;
  double wq[N];                 // 1D quadrature weights on [0,1]
  KernelTables<N> tab;          // D / DT used (B is the identity)
};

// ZSMEM: where d/dzeta of the three coordinate fields waits for the quadrature phase: in shared memory
// (3 more arrays per cell) or in 6(p+1) registers per thread.  Measured per degree (profiles/r1_v3_notes.md 7):
// registers win except at p = 5, 6, where they cost the third CTA per SM.
template <int P> struct OtfZInSmem { static constexpr bool value = (P == 5 || P == 6); };

template <int P, int CPT>
struct ApplyOtfCfg {
  static constexpr int N = P + 1, N2 = N * N, N3 = N2 * N;
  using L = SmemLayout<N, CPT>;
  static constexpr int ACTIVE = CPT * N2;
  static constexpr int NT = ((ACTIVE + 31) / 32) * 32;
  static constexpr int FIELD_DOUBLES = CPT * (2 * L::A_CS + L::B_CS);   // values + d/dxi (layout A), d/deta (layout B)
  // fields u, x, y, z; plus d/dzeta of x, y, z (written and read by the home thread only: keeping them in
  // registers across the line phase costs 6(p+1) registers and a CTA per SM)
  static constexpr bool ZSMEM = OtfZInSmem<P>::value;
  static constexpr size_t SMEM_BYTES = ((size_t)4 * FIELD_DOUBLES + (ZSMEM ? (size_t)3 * CPT * L::A_CS : 0)) * 8;
};

// OVERWRITE as in bp5_apply_kernel: 0 add, 1 store cell-interior DoFs, 2 = 1 + per-CTA partials of src.(A src)
template <int P, int CPT, int OVERWRITE>
__global__ void __launch_bounds__(ApplyOtfCfg<P, CPT>::NT)
    bp5_apply_otf_kernel(const __grid_constant__ ApplyOtfParams<P + 1> prm) {
  using Cfg = ApplyOtfCfg<P, CPT>;
  constexpr int N = Cfg::N, N2 = Cfg::N2;
  using L = typename Cfg::L;
  constexpr int A1 = L::A_S1, A2 = L::A_S2, B1 = L::B_S1, B2 = L::B_S2;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double *F = reinterpret_cast<double *>(smem_raw);      // [field][S0 | S1 | S2]
  constexpr int FS = Cfg::FIELD_DOUBLES, OS1 = CPT * L::A_CS, OS2 = 2 * CPT * L::A_CS;
  double *Z = F + 4 * FS;                                  // [3][CPT * A_CS]: d/dzeta of the coordinates
  constexpr int ZS = CPT * L::A_CS;

  if (prm.skip != nullptr && *prm.skip != 0) return;
  const int tid = threadIdx.x;
  const bool active = tid < Cfg::ACTIVE;
  const int c = active ? tid / N2 : 0;
  const int r = tid % N2;
  const int a = r % N, b = r / N;
  const int cA = c * L::A_CS, cB = c * L::B_CS;          // this cell's slice of an A / B array
  const double *__restrict__ Dx = prm.tab.D[0], *__restrict__ Dy = prm.tab.D[1], *__restrict__ Dz = prm.tab.D[2];
  const double *__restrict__ DTx = prm.tab.DT[0], *__restrict__ DTy = prm.tab.DT[1], *__restrict__ DTz = prm.tab.DT[2];
  const int ab_off = a + b * prm.sy;
  const int ab_irr = b * N + a;
  const int hA = b * A1 + a, hB = b * B1 + a;
  const int xA = b * A2 + a * A1;
  const int yA = b * A2 + a, yB = b * B2 + a;
  const double wab = prm.wq[a] * prm.wq[b];

  const long long tstride = gridDim.x;
  const long long n_tiles = prm.n_tiles;
  const int sz = prm.sz;
  const int *__restrict__ cell_base = prm.cell_base;
  const int *__restrict__ l2g_irr = prm.l2g_irr;
  double *__restrict__ dst = prm.dst;
  [[maybe_unused]] double dot_acc = 0.0;

  for (long long tile = prm.tile_begin + blockIdx.x; tile < n_tiles; tile += tstride) {
    const int base = active ? __ldg(cell_base + tile * CPT + c) : kNoCell;
    int idx[N];
    column_indices<N>(idx, l2g_irr, base, ab_off, ab_irr, sz);
    double t[N];             // d/dzeta of u along this thread's column, kept in registers to the end
    [[maybe_unused]] double tc[3][N];   // d/dzeta of x, y, z when they stay in registers
    // (1) home (i=a, j=b): gather the four columns, publish them, z-derivatives in registers
    {
      const double *__restrict__ fields[4] = {prm.src, prm.cx, prm.cy, prm.cz};
#pragma unroll
      for (int f = 0; f < 4; ++f) {
        double col[N];
#pragma unroll
        for (int k = 0; k < N; ++k) col[k] = (base == kNoCell) ? 0.0 : __ldg(fields[f] + idx[k]);
        if (active) {
          double *s0 = F + f * FS + cA;
#pragma unroll
          for (int k = 0; k < N; ++k) s0[hA + k * A2] = col[k];
          if (f == 0) contract_in_regs<N, -1>(t, Dz, col);
          else if constexpr (Cfg::ZSMEM) contract_to_smem<N, -1>(Z + (f - 1) * ZS + cA + hA, A2, Dz, col);
          else contract_in_regs<N, -1>(tc[f > 0 ? f - 1 : 0], Dz, col);
        }
      }
    }
    __syncthreads();
    // (2) x-line (j=a, k=b) and y-line (i=a, k=b): derivative along the line, one field after the other
    //     (rolled: the four fields share the code and the matrix operands)
    // the four fields (u, x, y, z) share the code; unrolled over the fields (four independent chains, ~60 more
    // registers) where it measured faster: p = 5 +11 %, p = 7 +11 %, p = 4 / 6 slower (profiles/r2_notes.md)
    if (active) {
      auto lines_of_field = [&](int f) {
        double *s0 = F + f * FS + cA, *s1 = F + f * FS + OS1 + cA, *s2 = F + f * FS + OS2 + cB;
        double v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = s0[xA + i];
        contract_to_smem<N, -1>(s1 + xA, 1, Dx, v);
#pragma unroll
        for (int j = 0; j < N; ++j) v[j] = s0[yA + j * A1];
        contract_to_smem<N, -1>(s2 + yB, B1, Dy, v);
      };
      if constexpr (P == 5 || P == 7) {
#pragma unroll
        for (int f = 0; f < 4; ++f) lines_of_field(f);
      } else {
#pragma unroll 1
        for (int f = 0; f < 4; ++f) lines_of_field(f);
      }
    }
    __syncthreads();
    // (3) quadrature-point phase (home): Jacobian from the coordinate gradients, G, g <- G g
    double *s1 = F + OS1 + cA, *s2 = F + OS2 + cB;       // the u field's derivative arrays
    if (active) {
#pragma unroll
      for (int k = 0; k < N; ++k) {
        const int wA = hA + k * A2, wB = hB + k * B2;
        double J[3][3];
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          J[d][0] = F[(d + 1) * FS + OS1 + cA + wA];
          J[d][1] = F[(d + 1) * FS + OS2 + cB + wB];
          if constexpr (Cfg::ZSMEM) J[d][2] = Z[d * ZS + cA + wA];
          else J[d][2] = tc[d][k];
        }
        // adj = det * J^-1 (rows: d xi_d / d x_f times det)
        const double a00 = J[1][1] * J[2][2] - J[1][2] * J[2][1], a01 = J[0][2] * J[2][1] - J[0][1] * J[2][2],
                     a02 = J[0][1] * J[1][2] - J[0][2] * J[1][1];
        const double a10 = J[1][2] * J[2][0] - J[1][0] * J[2][2], a11 = J[0][0] * J[2][2] - J[0][2] * J[2][0],
                     a12 = J[0][2] * J[1][0] - J[0][0] * J[1][2];
        const double a20 = J[1][0] * J[2][1] - J[1][1] * J[2][0], a21 = J[0][1] * J[2][0] - J[0][0] * J[2][1],
                     a22 = J[0][0] * J[1][1] - J[0][1] * J[1][0];
        const double det = J[0][0] * a00 + J[0][1] * a10 + J[0][2] * a20;
        const double sc = base == kNoCell ? 0.0 : wab * prm.wq[k] / det;   // JxW / det^2 (padding cells: no geometry)
        const double g0 = sc * (a00 * a00 + a01 * a01 + a02 * a02), g1 = sc * (a10 * a10 + a11 * a11 + a12 * a12),
                     g2 = sc * (a20 * a20 + a21 * a21 + a22 * a22);
        const double g3 = sc * (a00 * a10 + a01 * a11 + a02 * a12), g4 = sc * (a00 * a20 + a01 * a21 + a02 * a22),
                     g5 = sc * (a10 * a20 + a11 * a21 + a12 * a22);
        const double ur = s1[wA], us = s2[wB], ut = t[k];
        const double vr = ur * g0 + us * g3 + ut * g4;
        const double vs = ur * g3 + us * g1 + ut * g5;
        const double vt = ur * g4 + us * g5 + ut * g2;
        s1[wA] = vr;
        s2[wB] = vs;
        t[k] = vt;
        if constexpr (OVERWRITE == 2) dot_acc += ur * vr + us * vs + ut * vt;
      }
    }
    __syncthreads();
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
    if (base != kNoCell) {
      const bool col_interior = OVERWRITE != 0 && a > 0 && a < P && b > 0 && b < P;
      double o[N];
      contract_in_regs<N, -1>(o, DTz, t);
#pragma unroll
      for (int k = 0; k < N; ++k) {
        const double s = o[k] + s1[hA + k * A2] + s2[hB + k * B2];
        double *dp = dst + idx[k];
        if (col_interior && k > 0 && k < P) *dp = s;
        else atomicAdd(dp, s);
      }
    }
    // no barrier here: the next tile first writes the value arrays, which nobody reads any more
  }
  if constexpr (OVERWRITE == 2) {
    __syncthreads();
    double v = active ? dot_acc : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((tid & 31) == 0) F[tid >> 5] = v;
    __syncthreads();
    if (tid < 32) {
      v = tid < Cfg::NT / 32 ? F[tid] : 0.0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (tid == 0) prm.dot_partials[blockIdx.x] = v;
    }
  }
}

}  // namespace bp5
