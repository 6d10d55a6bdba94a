// Geometry on the fly for EVERY operator / quadrature combination (BASELINE config 5 for the reference's shipped
// default QGauss(p+1), bp5/step-64.cu:243-247, and for the Helmholtz operator of config 2,
// step-64/step-64.cu:201-219): nothing but the nodal coordinates of the degree-p mapped cells is stored
// (24 bytes per DoF, the support points of MappingQGeneric(p), bp5/step-64.cu:234) and the CTA REBUILDS the tile's
// coefficient in shared memory before it applies it:
//   for each coordinate field x_d: gather -> the same sum-factorised evaluation as the solution (values and
//   gradient at the quadrature points; Gauss: interpolate, then collocation derivative)
//     -> the line contractions write d x_d / d xi_e straight into a staged Jacobian (+ |x(q)|^2, Helmholtz only)
//   then the solution field; at every quadrature point
//     G = w_q / det(J) adj(J) adj(J)^T  (== JxW J^-1 J^-T, JacobianFunctor, bp5/step-64.cu:84-114)
//     a(x) JxW with a = 10 / (0.05 + 2 |x|^2)  (VaryingCoefficientFunctor, step-64/step-64.cu:100-118)
//   exactly what setup.cu:write_cell_metric stores, so the two geometry modes agree to rounding.
// Thread roles, shared-memory layouts, scatter and the fused src.(A src) are those of apply.cuh; four evaluations
// per tile instead of one make this a memory-saving mode: 0.52-0.59 of the stored-metric CG rate with a quarter of
// the geometry bytes (DESIGN.md 3.1b; ncu: shared-memory pipe 76 %, fp64 pipe 40 %).  The four-fields-at-once
// collocation kernel of apply_otf.cuh keeps p <= 4, the affine fast path of apply.cuh undeformed Poisson meshes.
// Algorithmic bytes: 16 (src, dst) + 24 (coordinates) per DoF.
#pragma once
#include "apply.cuh"

namespace bp5 {

template <int N>
struct ApplyOtfgParams {
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
  KernelTables<N> tab;
};

template <int P, int HELM, int CPT>
struct ApplyOtfgCfg {
  static constexpr int N = P + 1, N2 = N * N, N3 = N2 * N;
  using L = SmemLayout<N, CPT>;
  static constexpr int ACTIVE = CPT * N2;
  static constexpr int NT = ((ACTIVE + 31) / 32) * 32;
  // the staged Jacobian: d x_f / d xi in layout-A arrays and d x_f / d eta in layout-B arrays, written straight by
  // the line contractions of the coordinate fields; d x_f / d zeta (and |x|^2, Helmholtz) dense, private to the
  // home thread of the column
  static constexpr int JA_DOUBLES = 3 * CPT * L::A_CS, JB_DOUBLES = 3 * CPT * L::B_CS;
  static constexpr int JZ_PLANES = 3 + HELM;
  static constexpr int STAGE_DOUBLES = JA_DOUBLES + JB_DOUBLES + JZ_PLANES * CPT * N3;
  static constexpr int WORK_DOUBLES = CPT * (2 * L::A_CS + L::B_CS);    // S0, S1 (layout A), S2 (layout B)
  static constexpr size_t SMEM_BYTES = ((size_t)STAGE_DOUBLES + WORK_DOUBLES) * 8;
};

// QUAD, HELM, OVERWRITE as in bp5_apply_kernel (0 add, 1 store cell-interior DoFs, 2 = 1 + partials of src.(A src))
template <int P, int QUAD, int HELM, int CPT, int OVERWRITE>
__global__ void __launch_bounds__(ApplyOtfgCfg<P, HELM, CPT>::NT)
    bp5_apply_otfg_kernel(const __grid_constant__ ApplyOtfgParams<P + 1> prm) {
  using Cfg = ApplyOtfgCfg<P, HELM, CPT>;
  constexpr int N = Cfg::N, N2 = Cfg::N2, N3 = Cfg::N3;
  using L = typename Cfg::L;
  constexpr int A1 = L::A_S1, A2 = L::A_S2, B1 = L::B_S1, B2 = L::B_S2;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double *JA = reinterpret_cast<double *>(smem_raw);      // [3][CPT][A_CS]
  double *JB = JA + Cfg::JA_DOUBLES;                      // [3][CPT][B_CS]
  double *JZ = JB + Cfg::JB_DOUBLES;                      // [3 (+1)][CPT][N3]
  double *S0 = JA + Cfg::STAGE_DOUBLES;
  double *S1 = S0 + CPT * L::A_CS;
  double *S2 = S1 + CPT * L::A_CS;

  if (prm.skip != nullptr && *prm.skip != 0) return;
  const int tid = threadIdx.x;
  const bool active = tid < Cfg::ACTIVE;
  const int c = active ? tid / N2 : 0;
  const int r = tid % N2;
  const int a = r % N, b = r / N;
  double *s0 = S0 + c * L::A_CS, *s1 = S1 + c * L::A_CS, *s2 = S2 + c * L::B_CS;
  double *jz = JZ + c * N3 + b * N + a;                   // this thread's column: + field * CPT * N3 + k * N2
  const double *__restrict__ Bx = prm.tab.B[0], *__restrict__ By = prm.tab.B[1], *__restrict__ Bz = prm.tab.B[2];
  const double *__restrict__ BTx = prm.tab.BT[0], *__restrict__ BTy = prm.tab.BT[1], *__restrict__ BTz = prm.tab.BT[2];
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

  // values (mv, home column) and gradient (o1, layout A: d/dxi; o2, layout B: d/deta; t: d/dzeta in registers) of
  // one field at the quadrature points; the phases of bp5_apply_body.  Ends behind a barrier.
  auto evaluate = [&](const double (&u)[N], double (&t)[N], double (&mv)[N], double *o1, double *o2) {
    if constexpr (QUAD == 1) {
      if (active) {
#pragma unroll
        for (int k = 0; k < N; ++k) s0[hA + k * A2] = u[k];
        contract_in_regs<N, -1>(t, Dz, u);
#pragma unroll
        for (int k = 0; k < N; ++k) mv[k] = u[k];
      }
      __syncthreads();
      if (active) {
        double v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = s0[xA + i];
        contract_to_smem<N, -1>(o1 + xA, 1, Dx, v);
#pragma unroll
        for (int j = 0; j < N; ++j) v[j] = s0[yA + j * A1];
        contract_to_smem<N, -1>(o2 + yB, B1, Dy, v);
      }
      __syncthreads();
    } else {
      if (active) contract_to_smem<N, 1>(s0 + hA, A2, Bz, u);
      __syncthreads();
      if (active) {
        double v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = s0[xA + i];
        contract_to_smem<N, 1>(s0 + xA, 1, Bx, v);
      }
      __syncthreads();
      if (active) {
        double v[N], w[N];
#pragma unroll
        for (int j = 0; j < N; ++j) v[j] = s0[yA + j * A1];
        contract_in_regs<N, 1>(w, By, v);
#pragma unroll
        for (int q = 0; q < N; ++q) s0[yA + q * A1] = w[q];
        contract_to_smem<N, -1>(o2 + yB, B1, Dy, w);
      }
      __syncthreads();
      if (active) {
        double v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = s0[xA + i];
        contract_to_smem<N, -1>(o1 + xA, 1, Dx, v);
#pragma unroll
        for (int k = 0; k < N; ++k) mv[k] = s0[hA + k * A2];
        contract_in_regs<N, -1>(t, Dz, mv);
      }
      __syncthreads();
    }
  };

  // the gather of a field's columns is issued one evaluation ahead (the x coordinates of the next tile behind the
  // solution field of this one): its L2 latency hides behind the contractions of the field before (N more registers;
  // within +-5 % of gathering each field right before its evaluation, profiles/r2_otf_general_tuning.log)
  auto gather = [&](double (&v)[N], const double *__restrict__ fld, int bs) {
    int ix[N];
    column_indices<N>(ix, l2g_irr, bs, ab_off, ab_irr, sz);
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] = (bs == kNoCell) ? 0.0 : __ldg(fld + ix[k]);
  };
  long long tile = prm.tile_begin + blockIdx.x;
  int base = (active && tile < n_tiles) ? __ldg(cell_base + tile * CPT + c) : kNoCell;
  double col[N];
  gather(col, prm.cx, base);
  for (; tile < n_tiles; tile += tstride) {
    double t[N], mv[N], nxt[N];
    // ---------------- geometry: Jacobian (and |x|^2) of the tile's cells at the quadrature points -> stage
#pragma unroll 1
    for (int f = 0; f < 3; ++f) {
      gather(nxt, f == 0 ? prm.cy : f == 1 ? prm.cz : prm.src, base);
      evaluate(col, t, mv, JA + (f * CPT + c) * L::A_CS, JB + (f * CPT + c) * L::B_CS);
      if (active) {
        double *zp = jz + f * CPT * N3;
#pragma unroll
        for (int k = 0; k < N; ++k) {
          zp[k * N2] = t[k];
          if constexpr (HELM) {
            double *xp = jz + 3 * CPT * N3 + k * N2;
            *xp = (f == 0 ? 0.0 : *xp) + mv[k] * mv[k];
          }
        }
      }
#pragma unroll
      for (int k = 0; k < N; ++k) col[k] = nxt[k];
      // no barrier: the next evaluation first writes S0, which nobody reads any more
    }
    // ---------------- the solution field
    const int base_n = (active && tile + tstride < n_tiles) ? __ldg(cell_base + (tile + tstride) * CPT + c) : kNoCell;
    gather(nxt, prm.cx, base_n);
    evaluate(col, t, mv, s1, s2);
    // ---------------- quadrature-point phase (home): G from the staged Jacobian, g <- G g (+ mass term)
    if (active) {
#pragma unroll
      for (int k = 0; k < N; ++k) {
        const int wA = hA + k * A2, wB = hB + k * B2;
        double J[3][3];
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          J[d][0] = JA[(d * CPT + c) * L::A_CS + wA];
          J[d][1] = JB[(d * CPT + c) * L::B_CS + wB];
          J[d][2] = jz[d * CPT * N3 + k * N2];
        }
        // adj = det * J^-1 (rows: d xi_d / d x_f times det)
        const double a00 = J[1][1] * J[2][2] - J[1][2] * J[2][1], a01 = J[0][2] * J[2][1] - J[0][1] * J[2][2],
                     a02 = J[0][1] * J[1][2] - J[0][2] * J[1][1];
        const double a10 = J[1][2] * J[2][0] - J[1][0] * J[2][2], a11 = J[0][0] * J[2][2] - J[0][2] * J[2][0],
                     a12 = J[0][2] * J[1][0] - J[0][0] * J[1][2];
        const double a20 = J[1][0] * J[2][1] - J[1][1] * J[2][0], a21 = J[0][1] * J[2][0] - J[0][0] * J[2][1],
                     a22 = J[0][0] * J[1][1] - J[0][1] * J[1][0];
        const double det = J[0][0] * a00 + J[0][1] * a10 + J[0][2] * a20;
        const double w = wab * prm.wq[k];
        const double sc = base == kNoCell ? 0.0 : w / det;   // JxW / det^2 (padding cells: no geometry)
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
        if constexpr (HELM) {
          const double m_old = mv[k];
          mv[k] = m_old * (10.0 / (0.05 + 2.0 * jz[3 * CPT * N3 + k * N2]) * (w * det));
          if constexpr (OVERWRITE == 2) dot_acc += m_old * mv[k];
        }
      }
    }
    __syncthreads();
    // ---------------- integrate and scatter
    const bool col_interior = OVERWRITE != 0 && a > 0 && a < P && b > 0 && b < P;
    const bool do_scatter = base != kNoCell;
    int idx[N];
    column_indices<N>(idx, l2g_irr, base, ab_off, ab_irr, sz);
    if constexpr (QUAD == 1) {
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
      if (do_scatter) {
        double o[N];
        contract_in_regs<N, -1>(o, DTz, t);
#pragma unroll
        for (int k = 0; k < N; ++k) {
          double s = o[k] + s1[hA + k * A2] + s2[hB + k * B2];
          if constexpr (HELM) s += mv[k];
          double *dp = dst + idx[k];
          if (col_interior && k > 0 && k < P) *dp = s;
          else atomicAdd(dp, s);
        }
      }
    } else {
      if (active) {
        double v[N];
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = s1[xA + i];
        contract_to_smem<N, -1>(s1 + xA, 1, DTx, v);
        double o[N];
        contract_in_regs<N, -1>(o, DTz, t);
#pragma unroll
        for (int k = 0; k < N; ++k) s0[hA + k * A2] = HELM ? o[k] + mv[k] : o[k];
      }
      __syncthreads();
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
      if (active) {
        double v[N];
#pragma unroll
        for (int q = 0; q < N; ++q) v[q] = s0[xA + q];
        contract_to_smem<N, 1>(s0 + xA, 1, BTx, v);
      }
      __syncthreads();
      if (do_scatter) {
        double v[N], o[N];
#pragma unroll
        for (int q = 0; q < N; ++q) v[q] = s0[hA + q * A2];
        contract_in_regs<N, 1>(o, BTz, v);
#pragma unroll
        for (int k = 0; k < N; ++k) {
          double *dp = dst + idx[k];
          if (col_interior && k > 0 && k < P) *dp = o[k];
          else atomicAdd(dp, o[k]);
        }
      }
    }
    // no barrier here: the next tile first writes S0 -- the home columns (read last by their own threads) under
    // Gauss, an array nobody reads after the line phase under collocation
    base = base_n;
#pragma unroll
    for (int k = 0; k < N; ++k) col[k] = nxt[k];
  }
  if constexpr (OVERWRITE == 2) {
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

}  // namespace bp5
