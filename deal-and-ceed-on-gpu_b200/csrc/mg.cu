// Geometric multigrid on one block of a conforming structured mesh: a Chebyshev-Jacobi V-cycle as the
// preconditioner of a standard CG -- what deal.II users build from MGTransferMatrixFree, PreconditionChebyshev,
// MGCoarseGridIterativeSolver and PreconditionMG around a matrix-free operator [UPSTREAM].
//
//  * levels: the caller's operator, then the same problem with every cells[d] halved while all are even.  Each
//    level is an ordinary operator (tuned cell kernel, same geometry description).
//  * transfer: on one block the owned DoFs are the lexicographic lattice (p c_x + 1) x (p c_y + 1) x (p c_z + 1),
//    so nodal interpolation coarse -> fine is P_z (x) P_y (x) P_x with 1D matrices whose rows hold the
//    parent-to-child table l_b((s + xi_a) / 2).  It runs as three 1D passes; restriction is the exact transpose,
//    each output point gathering its inputs in a fixed order (no atomics: bitwise repeatable).
//  * smoother: Chebyshev iteration with D^-1 (Saad, Alg. 12.1); after each operator application one fused
//    streaming kernel does r -= t, d = a d + c D^-1 r, x += d.
//  * coarse level: cg_solve (standard CG, Jacobi) to a relative tolerance.
//  * outer solver: preconditioned standard CG with host scalars (about ten iterations, each one V-cycle).
#include <algorithm>
#include <array>
#include <cmath>
#include <vector>

#include "apply.cuh"
#include "cg_state.cuh"
#include "common.h"

namespace bp5 {

// ---------------------------------------------------------------- kernels
struct TransferPass {
  int p, c;                // degree; coarse cells along the pass direction
  int out_n[3];            // output lattice
  int in_n[3];             // input lattice (differs from out_n along the pass direction only)
  double H[2][kMaxN * kMaxN];   // parent-to-child table [s][a * n + b]
};

template <int DIR>
__device__ __forceinline__ void pass_coords(const TransferPass &prm, long long t, int &f, long long &base,
                                            long long &stride) {
  const int i0 = (int)(t % prm.out_n[0]);
  const long long rest = t / prm.out_n[0];
  const int i1 = (int)(rest % prm.out_n[1]), i2 = (int)(rest / prm.out_n[1]);
  const long long s1 = prm.in_n[0], s2 = (long long)prm.in_n[0] * prm.in_n[1];
  if (DIR == 0) { f = i0; base = s1 * i1 + s2 * i2; stride = 1; }
  else if (DIR == 1) { f = i1; base = i0 + s2 * i2; stride = s1; }
  else { f = i2; base = i0 + s1 * i1; stride = s2; }
}

// Prolongation along DIR: fine point f (output) = sum_b H[s][a n + b] in[coarse node cc p + b], where fine cell
// fc = min(f / p, 2c - 1) is child s = fc % 2 of coarse cell cc = fc / 2 and a = f - fc p.  ADD: out += P in.
template <int DIR, bool ADD>
__global__ void __launch_bounds__(256) mg_prolongate_1d(const __grid_constant__ TransferPass prm,
                                                        const double *__restrict__ in, double *__restrict__ out,
                                                        long long n_out) {
  const int p = prm.p, n = p + 1;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n_out; t += (long long)gridDim.x * blockDim.x) {
    int f;
    long long base, stride;
    pass_coords<DIR>(prm, t, f, base, stride);
    const int fc = min(f / p, 2 * prm.c - 1), a = f - fc * p, s = fc & 1;
    const double *src = in + base + (long long)(fc >> 1) * p * stride;
    const double *h = &prm.H[s][a * n];
    double v = 0.0;
    for (int b = 0; b < n; ++b) v += h[b] * src[b * stride];
    if (ADD) out[t] += v;
    else out[t] = v;
  }
}

// Restriction along DIR, the transpose of mg_prolongate_1d: coarse node j gathers every fine row whose owning fine
// cell (rows a = 0..p-1 of each fine cell, and a = p of the last one) is a child of a coarse cell containing j.
template <int DIR>
__global__ void __launch_bounds__(256) mg_restrict_1d(const __grid_constant__ TransferPass prm,
                                                      const double *__restrict__ in, double *__restrict__ out,
                                                      long long n_out) {
  const int p = prm.p, n = p + 1, c = prm.c;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n_out; t += (long long)gridDim.x * blockDim.x) {
    int j;
    long long base, stride;
    pass_coords<DIR>(prm, t, j, base, stride);
    const int cc_lo = (j % p == 0 && j > 0) ? j / p - 1 : j / p, cc_hi = min(j / p, c - 1);
    double v = 0.0;
#pragma unroll 1
    for (int cc = cc_lo; cc <= cc_hi; ++cc) {
      const int b = j - cc * p;
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        const int fc = 2 * cc + s, amax = (fc == 2 * c - 1) ? p : p - 1;
        const double *src = in + base + (long long)fc * p * stride;
        for (int a = 0; a <= amax; ++a) v += prm.H[s][a * n + b] * src[a * stride];
      }
    }
    out[t] = v;
  }
}

// Dirichlet rows of a restricted vector: v[list[i]] = 0 (the level operator's constrained list)
__global__ void mg_zero_constrained(const int *__restrict__ list, long long n, double *__restrict__ v) {
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (t < n) v[list[t]] = 0.0;
}

// One Chebyshev step after the operator application t = A (.):
//   MODE 0 (start from x = 0, no t):  d = c D^-1 rsrc;  x = d
//   MODE 1 (step):                    r = rsrc - t;  d = a d + c D^-1 r  (a == 0: d not read);  x += d
//   MODE 2 (residual only):           r = rsrc - t
template <int MODE>
__global__ void __launch_bounds__(256) mg_chebyshev_step(const double *rsrc, const double *__restrict__ t,
                                                         double *r, double *__restrict__ d, double *__restrict__ x,
                                                         const double *__restrict__ dinv, double a, double c,
                                                         long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    if (MODE == 0) {
      const double dn = c * dinv[i] * rsrc[i];
      d[i] = dn;
      x[i] = dn;
    } else {
      const double rn = rsrc[i] - t[i];
      r[i] = rn;
      if (MODE == 1) {
        const double dn = (a == 0.0 ? 0.0 : a * d[i]) + c * dinv[i] * rn;
        d[i] = dn;
        x[i] += dn;
      }
    }
  }
}

// fixed-seed start vector of the eigenvalue estimate: uniform in [-1, 1) from a hash of the index
__global__ void mg_random_fill(double *__restrict__ v, long long n, unsigned long long seed) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    unsigned long long z = seed + 0x9e3779b97f4a7c15ull * (unsigned long long)(i + 1);
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    z ^= z >> 31;
    v[i] = (double)(z >> 11) * (2.0 / 9007199254740992.0) - 1.0;
  }
}

static unsigned mg_grid(long long n, int sm_count) {
  long long g = (n + 255) / 256;
  const long long cap = (long long)sm_count * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (unsigned)g;
}

}  // namespace bp5

using namespace bp5;

// ---------------------------------------------------------------- object
struct bp5_mg_s {
  struct Level {
    bp5_operator_t op = nullptr;
    bool owned = false;
    int cells[3] = {0, 0, 0}, nd[3] = {0, 0, 0};
    int64_t n = 0;
    bp5_vector_t b = nullptr, x = nullptr;            // coarser levels: right-hand side and solution of V_l
    bp5_vector_t r = nullptr, d = nullptr, t = nullptr, dinv = nullptr;
    double *s1 = nullptr, *s2 = nullptr;              // levels >= 1: intermediate lattices of the 1D transfer passes
    double lambda = 0.0;                              // estimate of lambda_max(D^-1 A), levels >= 1
  };
  bp5_context_t ctx = nullptr;
  int degree = 5, eig_its = 12, coarse_max_its = 1000, n_levels = 0;
  double range = 15.0, coarse_tol = 1e-6;
  std::vector<Level> lv;
  TransferPass pass{};                                // p and H; the lattice fields are set per pass
  bp5_vector_t g = nullptr, h = nullptr, dd = nullptr, ad = nullptr;   // outer CG
  // profiling: event pairs tagged with (level, category)
  bool profile = false;
  std::vector<cudaEvent_t> ev;
  std::vector<int> ev_tag;
  size_t ev_used = 0;
  int64_t n_vcycles = 0;
  std::vector<double> prof_ms;
};

namespace bp5 {
namespace {

struct ProfScope {
  bp5_mg_t mg;
  size_t slot = (size_t)-1;
  ProfScope(bp5_mg_t m, int level, int cat) : mg(m) {
    if (!mg->profile) return;
    if (mg->ev_used + 2 > mg->ev.size()) {
      cudaEvent_t a, b;
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return;
      mg->ev.push_back(a); mg->ev.push_back(b);
      mg->ev_tag.push_back(0);
    }
    slot = mg->ev_used;
    mg->ev_tag[slot / 2] = 4 * level + cat;
    mg->ev_used += 2;
    cudaEventRecord(mg->ev[slot], mg->ctx->stream);
  }
  ~ProfScope() {
    if (slot != (size_t)-1) cudaEventRecord(mg->ev[slot + 1], mg->ctx->stream);
  }
};

int prof_collect(bp5_mg_t mg) {
  if (mg->ev_used == 0) return BP5_OK;
  BP5_CUDA(cudaStreamSynchronize(mg->ctx->stream));
  for (size_t k = 0; k < mg->ev_used; k += 2) {
    float ms = 0.f;
    BP5_CUDA(cudaEventElapsedTime(&ms, mg->ev[k], mg->ev[k + 1]));
    mg->prof_ms[mg->ev_tag[k / 2]] += ms;
  }
  mg->ev_used = 0;
  return BP5_OK;
}

// A src on a level (Dirichlet rows: identity), independent of the operator's do_zero_out
int level_vmult(bp5_mg_t mg, int l, double *dst, const double *src) {
  ProfScope ps(mg, l, 0);
  bp5_operator_t op = mg->lv[l].op;
  int rc;
  if ((rc = apply_zero_skeleton(op, dst))) return rc;
  if ((rc = apply_cell_loop(op, dst, src, true))) return rc;
  return apply_copy_constrained(op, dst, src);
}

template <int MODE>
int cheb_kernel(bp5_mg_t mg, int l, const double *rsrc, const double *t, double *r, double *d, double *x, double a,
                double c) {
  ProfScope ps(mg, l, 2);
  const bp5_mg_s::Level &L = mg->lv[l];
  mg_chebyshev_step<MODE><<<mg_grid(L.n, mg->ctx->sm_count), 256, 0, mg->ctx->stream>>>(rsrc, t, r, d, x, L.dinv->d,
                                                                                        a, c, L.n);
  BP5_CHECK_LAUNCH();
  mg->ctx->launches++;
  return BP5_OK;
}

// x <- Chebyshev smoothing of A x = b on level l >= 1 (x_zero: x == 0 on entry, not read)
int smooth(bp5_mg_t mg, int l, double *x, const double *b, bool x_zero) {
  bp5_mg_s::Level &L = mg->lv[l];
  const double lmax = 1.2 * L.lambda, lmin = lmax / mg->range;
  const double theta = 0.5 * (lmax + lmin), delta = 0.5 * (lmax - lmin), sigma = theta / delta;
  double rho0 = 1.0 / sigma;
  double *r = L.r->d, *d = L.d->d, *t = L.t->d;
  int rc;
  if (x_zero) {
    if ((rc = cheb_kernel<0>(mg, l, b, nullptr, nullptr, d, x, 0.0, 1.0 / theta))) return rc;
  } else {
    if ((rc = level_vmult(mg, l, t, x))) return rc;
    if ((rc = cheb_kernel<1>(mg, l, b, t, r, d, x, 0.0, 1.0 / theta))) return rc;
  }
  for (int j = 2; j <= mg->degree; ++j) {
    if ((rc = level_vmult(mg, l, t, d))) return rc;
    const double rho1 = 1.0 / (2.0 * sigma - rho0);
    const double *rsrc = (j == 2 && x_zero) ? b : r;
    if ((rc = cheb_kernel<1>(mg, l, rsrc, t, r, d, x, rho1 * rho0, 2.0 * rho1 / delta))) return rc;
    rho0 = rho1;
  }
  return BP5_OK;
}

int transfer_launch(bp5_mg_t mg, int fine_level, bool restrict_, int dir, bool add, const double *in, double *out) {
  const bp5_mg_s::Level &F = mg->lv[fine_level], &Cl = mg->lv[fine_level - 1];
  TransferPass &prm = mg->pass;
  // prolongation runs x, y, z: C -> (F C C) -> (F F C) -> F; restriction runs z, y, x: F -> (F F C) -> (F C C) -> C
  for (int e = 0; e < 3; ++e) {
    const bool fine_in = restrict_ ? e <= dir : e < dir;
    const bool fine_out = restrict_ ? e < dir : e <= dir;
    prm.in_n[e] = fine_in ? F.nd[e] : Cl.nd[e];
    prm.out_n[e] = fine_out ? F.nd[e] : Cl.nd[e];
  }
  prm.c = Cl.cells[dir];
  const long long n_out = (long long)prm.out_n[0] * prm.out_n[1] * prm.out_n[2];
  const unsigned grid = mg_grid(n_out, mg->ctx->sm_count);
  cudaStream_t s = mg->ctx->stream;
  if (restrict_) {
    if (dir == 0) mg_restrict_1d<0><<<grid, 256, 0, s>>>(prm, in, out, n_out);
    else if (dir == 1) mg_restrict_1d<1><<<grid, 256, 0, s>>>(prm, in, out, n_out);
    else mg_restrict_1d<2><<<grid, 256, 0, s>>>(prm, in, out, n_out);
  } else if (add) {
    if (dir == 0) mg_prolongate_1d<0, true><<<grid, 256, 0, s>>>(prm, in, out, n_out);
    else if (dir == 1) mg_prolongate_1d<1, true><<<grid, 256, 0, s>>>(prm, in, out, n_out);
    else mg_prolongate_1d<2, true><<<grid, 256, 0, s>>>(prm, in, out, n_out);
  } else {
    if (dir == 0) mg_prolongate_1d<0, false><<<grid, 256, 0, s>>>(prm, in, out, n_out);
    else if (dir == 1) mg_prolongate_1d<1, false><<<grid, 256, 0, s>>>(prm, in, out, n_out);
    else mg_prolongate_1d<2, false><<<grid, 256, 0, s>>>(prm, in, out, n_out);
  }
  BP5_CHECK_LAUNCH();
  mg->ctx->launches++;
  return BP5_OK;
}

// dst (level fine_level) = P src, or += P src
int prolongate(bp5_mg_t mg, int fine_level, double *dst, const double *src, bool add) {
  ProfScope ps(mg, fine_level, 1);
  const bp5_mg_s::Level &F = mg->lv[fine_level];
  int rc;
  if ((rc = transfer_launch(mg, fine_level, false, 0, false, src, F.s1))) return rc;
  if ((rc = transfer_launch(mg, fine_level, false, 1, false, F.s1, F.s2))) return rc;
  return transfer_launch(mg, fine_level, false, 2, add, F.s2, dst);
}

// dst (level fine_level-1) = R src, Dirichlet rows zeroed
int restrict_(bp5_mg_t mg, int fine_level, double *dst, const double *src) {
  ProfScope ps(mg, fine_level, 1);
  const bp5_mg_s::Level &F = mg->lv[fine_level];
  int rc;
  if ((rc = transfer_launch(mg, fine_level, true, 2, false, src, F.s2))) return rc;
  if ((rc = transfer_launch(mg, fine_level, true, 1, false, F.s2, F.s1))) return rc;
  if ((rc = transfer_launch(mg, fine_level, true, 0, false, F.s1, dst))) return rc;
  bp5_operator_t cop = mg->lv[fine_level - 1].op;
  if (cop->n_constrained > 0) {
    const long long nc = cop->n_constrained;
    mg_zero_constrained<<<(unsigned)((nc + 255) / 256), 256, 0, mg->ctx->stream>>>(cop->constrained, nc, dst);
    BP5_CHECK_LAUNCH();
    mg->ctx->launches++;
  }
  return BP5_OK;
}

int coarse_solve(bp5_mg_t mg, bp5_vector_t x, bp5_vector_t b) {
  ProfScope ps(mg, 0, 3);
  bp5_mg_s::Level &L = mg->lv[0];
  int rc;
  if ((rc = vec_fill(mg->ctx, x->d, L.n, 0.0))) return rc;
  double bb = 0.0;
  if ((rc = vec_dot(mg->ctx, b->d, b->d, L.n, &bb))) return rc;
  int its = 0;
  double res = 0.0;
  rc = cg_solve(L.op, x, b, L.dinv, BP5_CG_STANDARD, BP5_CONTROL_ITERATION_NUMBER, mg->coarse_tol * std::sqrt(bb),
                mg->coarse_max_its, &its, &res, nullptr, 0);
  if (rc == BP5_ERR_NO_CONVERGENCE) rc = BP5_OK;   // x holds the last iterate: fine for a preconditioner
  return rc;
}

// x = V_l(b), from a zero initial guess
int vcycle(bp5_mg_t mg, int l, bp5_vector_t x, bp5_vector_t b) {
  if (l == 0) return coarse_solve(mg, x, b);
  bp5_mg_s::Level &L = mg->lv[l], &C = mg->lv[l - 1];
  int rc;
  if ((rc = smooth(mg, l, x->d, b->d, true))) return rc;                          // 1. pre-smooth from 0
  if ((rc = level_vmult(mg, l, L.t->d, x->d))) return rc;                          // 2. r = b - A x
  if ((rc = cheb_kernel<2>(mg, l, b->d, L.t->d, L.r->d, nullptr, nullptr, 0.0, 0.0))) return rc;
  if ((rc = restrict_(mg, l, C.b->d, L.r->d))) return rc;                          // 3. b_{l-1} = R r
  if ((rc = vcycle(mg, l - 1, C.x, C.b))) return rc;                               // 4. x += P V_{l-1}
  if ((rc = prolongate(mg, l, x->d, C.x->d, true))) return rc;
  return smooth(mg, l, x->d, b->d, false);                                         // 5. post-smooth
}

// lambda_max(D^-1 A) on level l by `eig_its` steps of Jacobi-preconditioned CG (the Lanczos tridiagonal of the CG
// coefficients), from the fixed-seed vector with zero Dirichlet entries -- PreconditionChebyshev's estimate
int estimate_lambda(bp5_mg_t mg, int l, double *lambda) {
  bp5_mg_s::Level &L = mg->lv[l];
  bp5_context_t ctx = mg->ctx;
  const int64_t n = L.n;
  double *r = L.r->d, *z = L.d->d, *q = L.t->d, *p = L.x ? L.x->d : nullptr;
  bp5_vector_t pv = nullptr;
  int rc;
  if (!p) {   // finest level: no level-owned x, borrow a temporary
    if ((rc = bp5_vector_create(ctx, n, 0, &pv))) return rc;
    p = pv->d;
  }
  auto body = [&]() -> int {
    int rc;
    mg_random_fill<<<mg_grid(n, ctx->sm_count), 256, 0, ctx->stream>>>(r, n, 0x5eedull + (unsigned long long)l);
    BP5_CHECK_LAUNCH();
    ctx->launches++;
    if (L.op->n_constrained > 0) {
      mg_zero_constrained<<<(unsigned)((L.op->n_constrained + 255) / 256), 256, 0, ctx->stream>>>(
          L.op->constrained, L.op->n_constrained, r);
      BP5_CHECK_LAUNCH();
      ctx->launches++;
    }
    // z = D^-1 r ; p = z
    if ((rc = vec_axpy(ctx, z, 0.0, 1.0, r, n, 1))) return rc;
    if ((rc = vec_axpy(ctx, z, 0.0, 0.0, L.dinv->d, n, 3))) return rc;
    if ((rc = vec_axpy(ctx, p, 0.0, 1.0, z, n, 1))) return rc;
    double rz = 0.0;
    if ((rc = vec_dot(ctx, r, z, n, &rz))) return rc;
    std::vector<double> alpha, beta;
    for (int j = 0; j < mg->eig_its && rz > 0.0; ++j) {
      if ((rc = level_vmult(mg, l, q, p))) return rc;
      double pq = 0.0;
      if ((rc = vec_dot(ctx, p, q, n, &pq))) return rc;
      if (!(pq > 0.0)) break;
      const double a = rz / pq;
      alpha.push_back(a);
      if ((rc = vec_axpy(ctx, r, 0.0, -a, q, n, 0))) return rc;
      if ((rc = vec_axpy(ctx, z, 0.0, 1.0, r, n, 1))) return rc;
      if ((rc = vec_axpy(ctx, z, 0.0, 0.0, L.dinv->d, n, 3))) return rc;
      double rz_new = 0.0;
      if ((rc = vec_dot(ctx, r, z, n, &rz_new))) return rc;
      const double bt = rz_new / rz;
      rz = rz_new;
      if (j + 1 < mg->eig_its && rz > 0.0) {
        beta.push_back(bt);
        if ((rc = vec_axpy(ctx, p, bt, 1.0, z, n, 2))) return rc;
      }
    }
    BP5_REQUIRE(!alpha.empty(), "eigenvalue estimate: no CG step possible (zero start vector or operator)");
    // T[j][j] = 1/alpha_j + beta_{j-1}/alpha_{j-1}, T[j][j+1] = sqrt(beta_j)/alpha_j; largest eigenvalue by
    // bisection on Sturm counts inside the Gershgorin interval
    const int m = (int)alpha.size();
    std::vector<double> dg(m), off(m, 0.0);
    for (int j = 0; j < m; ++j) {
      dg[j] = 1.0 / alpha[j] + (j > 0 ? beta[j - 1] / alpha[j - 1] : 0.0);
      if (j + 1 < m) off[j] = std::sqrt(beta[j]) / alpha[j];
    }
    double lo = 0.0, hi = 0.0;
    for (int j = 0; j < m; ++j) {
      const double rad = std::fabs(off[j]) + (j > 0 ? std::fabs(off[j - 1]) : 0.0);
      hi = std::max(hi, dg[j] + rad);
    }
    auto count_above = [&](double x) {   // eigenvalues > x
      int cnt = 0;
      double dval = 1.0;
      for (int j = 0; j < m; ++j) {
        dval = dg[j] - x - (j > 0 ? off[j - 1] * off[j - 1] / dval : 0.0);
        if (dval == 0.0) dval = -1e-300;
        if (dval < 0.0) ++cnt;
      }
      return m - cnt;
    };
    for (int it = 0; it < 200 && hi - lo > 1e-15 * hi; ++it) {
      const double mid = 0.5 * (lo + hi);
      if (count_above(mid) > 0) lo = mid;
      else hi = mid;
    }
    *lambda = 0.5 * (lo + hi);
    return BP5_OK;
  };
  rc = body();
  if (pv) bp5_vector_destroy(pv);
  return rc;
}

int mg_check_level_vec(bp5_mg_t mg, int level, bp5_vector_t v) {
  BP5_REQUIRE(v != nullptr, "null vector");
  BP5_REQUIRE(v->n_owned == mg->lv[level].n && v->n_ghost == 0, "vector layout does not match the level");
  return BP5_OK;
}

void mg_free(bp5_mg_t mg) {
  if (!mg) return;
  cudaStreamSynchronize(mg->ctx->stream);
  for (auto &L : mg->lv) {
    bp5_vector_destroy(L.b); bp5_vector_destroy(L.x); bp5_vector_destroy(L.r); bp5_vector_destroy(L.d);
    bp5_vector_destroy(L.t); bp5_vector_destroy(L.dinv);
    cudaFree(L.s1); cudaFree(L.s2);
    if (L.owned) bp5_operator_destroy(L.op);
  }
  bp5_vector_destroy(mg->g); bp5_vector_destroy(mg->h); bp5_vector_destroy(mg->dd); bp5_vector_destroy(mg->ad);
  for (cudaEvent_t e : mg->ev) cudaEventDestroy(e);
  delete mg;
}

}  // namespace
}  // namespace bp5

#define BP5_MG_GUARD_BEGIN try {
#define BP5_MG_GUARD_END                                      \
  }                                                           \
  catch (const std::bad_alloc &) {                            \
    set_error("out of host memory");                          \
    return BP5_ERR_INVALID;                                   \
  }                                                           \
  catch (...) {                                               \
    set_error("unexpected C++ exception at the ABI boundary"); \
    return BP5_ERR_INVALID;                                   \
  }

extern "C" {

int bp5_mg_create(bp5_operator_t fine, const bp5_mg_params_t *params, bp5_mg_t *out) {
  BP5_MG_GUARD_BEGIN
  BP5_REQUIRE(fine && out, "null argument");
  bp5_mg_params_t prm{};
  if (params) prm = *params;
  for (int k = 0; k < 4; ++k) BP5_REQUIRE(prm.reserved[k] == 0, "reserved fields of bp5_mg_params_t must be zero");
  BP5_REQUIRE(prm.max_levels >= 0 && prm.smoothing_degree >= 0 && prm.eig_iterations >= 0 && prm.coarse_max_its >= 0,
              "multigrid parameters must be >= 0 (0: default)");
  BP5_REQUIRE(prm.smoothing_range >= 0.0 && prm.coarse_tol >= 0.0, "multigrid parameters must be >= 0 (0: default)");
  BP5_REQUIRE(prm.smoothing_range == 0.0 || prm.smoothing_range > 1.0, "smoothing_range must exceed 1");
  const bp5_problem_t &pr = fine->prob;
  if (fine->hanging || fine->n_ghost != 0 || pr.part_grid[0] * pr.part_grid[1] * pr.part_grid[2] != 1 ||
      pr.geometry_mode != BP5_GEOM_STORED || pr.cell_order != BP5_CELL_ORDER_DEFAULT) {
    set_error("multigrid is implemented for one block of a conforming mesh with stored geometry and the default "
              "cell order");
    return BP5_ERR_UNSUPPORTED;
  }
  bp5_context_t ctx = fine->ctx;
  BP5_CUDA(cudaSetDevice(ctx->device));
  bp5_mg_t mg = new bp5_mg_s;
  mg->ctx = ctx;
  if (prm.smoothing_degree) mg->degree = prm.smoothing_degree;
  if (prm.smoothing_range > 0.0) mg->range = prm.smoothing_range;
  if (prm.eig_iterations) mg->eig_its = prm.eig_iterations;
  if (prm.coarse_max_its) mg->coarse_max_its = prm.coarse_max_its;
  if (prm.coarse_tol > 0.0) mg->coarse_tol = prm.coarse_tol;
  // level cell counts, finest first
  std::vector<std::array<int, 3>> cells{{pr.cells[0], pr.cells[1], pr.cells[2]}};
  while (prm.max_levels == 0 || (int)cells.size() < prm.max_levels) {
    const auto &c = cells.back();
    if (c[0] % 2 || c[1] % 2 || c[2] % 2) break;
    cells.push_back({c[0] / 2, c[1] / 2, c[2] / 2});
  }
  mg->n_levels = (int)cells.size();
  mg->lv.resize(mg->n_levels);
  int rc = BP5_OK;
  for (int l = 0; l < mg->n_levels && rc == BP5_OK; ++l) {
    bp5_mg_s::Level &L = mg->lv[l];
    const auto &c = cells[mg->n_levels - 1 - l];
    if (l == mg->n_levels - 1) {
      L.op = fine;
    } else {
      bp5_problem_t q = pr;
      for (int d = 0; d < 3; ++d) q.cells[d] = c[d];
      if ((rc = bp5_operator_create(ctx, &q, &L.op))) break;
      L.owned = true;
    }
    for (int d = 0; d < 3; ++d) { L.cells[d] = c[d]; L.nd[d] = c[d] * pr.degree + 1; }
    L.n = L.op->n_owned;
    const int64_t n = L.n;
    if (l < mg->n_levels - 1) {
      if ((rc = bp5_vector_create(ctx, n, 0, &L.b))) break;
      if ((rc = bp5_vector_create(ctx, n, 0, &L.x))) break;
    }
    if (l > 0) {
      if ((rc = bp5_vector_create(ctx, n, 0, &L.r))) break;
      if ((rc = bp5_vector_create(ctx, n, 0, &L.d))) break;
      if ((rc = bp5_vector_create(ctx, n, 0, &L.t))) break;
      const auto &cc = cells[mg->n_levels - l];   // next coarser level
      const int64_t ncd[3] = {(int64_t)cc[0] * pr.degree + 1, (int64_t)cc[1] * pr.degree + 1,
                              (int64_t)cc[2] * pr.degree + 1};
      if (cudaMalloc(&L.s1, sizeof(double) * L.nd[0] * ncd[1] * ncd[2]) != cudaSuccess ||
          cudaMalloc(&L.s2, sizeof(double) * L.nd[0] * L.nd[1] * ncd[2]) != cudaSuccess) {
        set_error("cudaMalloc of the transfer scratch failed: %s", cudaGetErrorString(cudaGetLastError()));
        rc = BP5_ERR_CUDA;
        break;
      }
    }
    if ((rc = bp5_vector_create(ctx, n, 0, &L.dinv))) break;
    if ((rc = operator_diagonal(L.op, L.dinv->d, true))) break;
  }
  if (rc == BP5_OK) {
    mg->pass.p = pr.degree;
    parent_child_interp(fine->tab, mg->pass.H);
    for (int l = 1; l < mg->n_levels && rc == BP5_OK; ++l) rc = estimate_lambda(mg, l, &mg->lv[l].lambda);
  }
  if (rc == BP5_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
    set_error("multigrid set-up failed: %s", cudaGetErrorString(cudaGetLastError()));
    rc = BP5_ERR_CUDA;
  }
  if (rc != BP5_OK) {
    const std::string msg = get_error();   // keep the first error across the clean-up
    mg_free(mg);
    set_error("%s", msg.c_str());
    return rc;
  }
  mg->prof_ms.assign(4 * mg->n_levels, 0.0);
  *out = mg;
  return BP5_OK;
  BP5_MG_GUARD_END
}

int bp5_mg_destroy(bp5_mg_t mg) {
  if (!mg) return BP5_OK;
  cudaSetDevice(mg->ctx->device);
  mg_free(mg);
  return BP5_OK;
}

int bp5_mg_n_levels(bp5_mg_t mg, int *n_levels) {
  BP5_REQUIRE(mg && n_levels, "null argument");
  *n_levels = mg->n_levels;
  return BP5_OK;
}

int bp5_mg_level_operator(bp5_mg_t mg, int level, bp5_operator_t *op) {
  BP5_REQUIRE(mg && op, "null argument");
  BP5_REQUIRE(level >= 0 && level < mg->n_levels, "level out of range");
  *op = mg->lv[level].op;
  return BP5_OK;
}

int bp5_mg_get_lambda_max(bp5_mg_t mg, int level, double *lambda) {
  BP5_REQUIRE(mg && lambda, "null argument");
  BP5_REQUIRE(level >= 1 && level < mg->n_levels, "level out of range (level 0 is solved, not smoothed)");
  *lambda = mg->lv[level].lambda;
  return BP5_OK;
}

int bp5_mg_set_lambda_max(bp5_mg_t mg, int level, double lambda) {
  BP5_REQUIRE(mg, "null argument");
  BP5_REQUIRE(level >= 1 && level < mg->n_levels, "level out of range (level 0 is solved, not smoothed)");
  BP5_REQUIRE(lambda > 0.0 && std::isfinite(lambda), "lambda must be positive and finite");
  mg->lv[level].lambda = lambda;
  return BP5_OK;
}

int bp5_mg_prolongate(bp5_mg_t mg, int fine_level, bp5_vector_t dst, bp5_vector_t src) {
  BP5_MG_GUARD_BEGIN
  BP5_REQUIRE(mg, "null argument");
  BP5_REQUIRE(fine_level >= 1 && fine_level < mg->n_levels, "fine_level out of range");
  int rc;
  if ((rc = mg_check_level_vec(mg, fine_level, dst)) || (rc = mg_check_level_vec(mg, fine_level - 1, src))) return rc;
  BP5_CUDA(cudaSetDevice(mg->ctx->device));
  return prolongate(mg, fine_level, dst->d, src->d, false);
  BP5_MG_GUARD_END
}

int bp5_mg_restrict(bp5_mg_t mg, int fine_level, bp5_vector_t dst, bp5_vector_t src) {
  BP5_MG_GUARD_BEGIN
  BP5_REQUIRE(mg, "null argument");
  BP5_REQUIRE(fine_level >= 1 && fine_level < mg->n_levels, "fine_level out of range");
  int rc;
  if ((rc = mg_check_level_vec(mg, fine_level - 1, dst)) || (rc = mg_check_level_vec(mg, fine_level, src))) return rc;
  BP5_CUDA(cudaSetDevice(mg->ctx->device));
  return restrict_(mg, fine_level, dst->d, src->d);
  BP5_MG_GUARD_END
}

int bp5_mg_smooth(bp5_mg_t mg, int level, bp5_vector_t x, bp5_vector_t b) {
  BP5_MG_GUARD_BEGIN
  BP5_REQUIRE(mg, "null argument");
  BP5_REQUIRE(level >= 1 && level < mg->n_levels, "level out of range (level 0 is solved, not smoothed)");
  int rc;
  if ((rc = mg_check_level_vec(mg, level, x)) || (rc = mg_check_level_vec(mg, level, b))) return rc;
  BP5_REQUIRE(x != b, "x and b must differ");
  BP5_CUDA(cudaSetDevice(mg->ctx->device));
  int x_zero = 0;
  if ((rc = vec_all_zero(mg->ctx, x->d, x->n_owned, &x_zero))) return rc;
  return smooth(mg, level, x->d, b->d, x_zero != 0);
  BP5_MG_GUARD_END
}

int bp5_mg_vcycle(bp5_mg_t mg, bp5_vector_t dst, bp5_vector_t src) {
  BP5_MG_GUARD_BEGIN
  BP5_REQUIRE(mg, "null argument");
  const int top = mg->n_levels - 1;
  int rc;
  if ((rc = mg_check_level_vec(mg, top, dst)) || (rc = mg_check_level_vec(mg, top, src))) return rc;
  BP5_REQUIRE(dst != src, "dst and src must differ");
  BP5_CUDA(cudaSetDevice(mg->ctx->device));
  if ((rc = vcycle(mg, top, dst, src))) return rc;
  if (mg->profile) mg->n_vcycles++;
  return BP5_OK;
  BP5_MG_GUARD_END
}

int bp5_mg_cg_solve(bp5_mg_t mg, bp5_vector_t x, bp5_vector_t b, int control, double tol, int max_its, int *last_step,
                    double *last_value, double *history, int history_len) {
  BP5_MG_GUARD_BEGIN
  BP5_REQUIRE(mg, "null argument");
  const int top = mg->n_levels - 1;
  int rc;
  if ((rc = mg_check_level_vec(mg, top, x)) || (rc = mg_check_level_vec(mg, top, b))) return rc;
  BP5_REQUIRE(x != b, "x and b must differ");
  BP5_REQUIRE(max_its >= 0, "max_its must be >= 0");
  BP5_REQUIRE(control == BP5_CONTROL_ITERATION_NUMBER || control == BP5_CONTROL_SOLVER, "unknown control");
  BP5_CUDA(cudaSetDevice(mg->ctx->device));
  bp5_context_t ctx = mg->ctx;
  const int64_t n = mg->lv[top].n;
  if (!mg->g) {
    if ((rc = bp5_vector_create(ctx, n, 0, &mg->g))) return rc;
    if ((rc = bp5_vector_create(ctx, n, 0, &mg->h))) return rc;
    if ((rc = bp5_vector_create(ctx, n, 0, &mg->dd))) return rc;
    if ((rc = bp5_vector_create(ctx, n, 0, &mg->ad))) return rc;
  }
  double *g = mg->g->d, *d = mg->dd->d, *ad = mg->ad->d;
  // SolverCG::solve [UPSTREAM]: g = A x - b (or -b for x == 0)
  int x_zero = 0;
  if ((rc = vec_all_zero(ctx, x->d, n, &x_zero))) return rc;
  if (!x_zero) {
    if ((rc = level_vmult(mg, top, g, x->d))) return rc;
    if ((rc = vec_axpy(ctx, g, 0.0, -1.0, b->d, n, 0))) return rc;
  } else if ((rc = vec_axpy(ctx, g, 0.0, -1.0, b->d, n, 1))) {
    return rc;
  }
  double gg = 0.0;
  if ((rc = vec_dot(ctx, g, g, n, &gg))) return rc;
  double res = std::sqrt(gg);
  if (history && history_len > 0) history[0] = res;
  int it = 0, conv = control_check(control, 0, max_its, res, tol);
  double gh = 0.0;
  if (conv == 0) {
    if ((rc = vcycle(mg, top, mg->h, mg->g))) return rc;       // h = M^-1 g
    if (mg->profile) mg->n_vcycles++;
    if ((rc = vec_axpy(ctx, d, 0.0, -1.0, mg->h->d, n, 1))) return rc;   // d = -h
    if ((rc = vec_dot(ctx, g, mg->h->d, n, &gh))) return rc;
  }
  while (conv == 0) {
    ++it;
    if ((rc = level_vmult(mg, top, ad, d))) return rc;
    double dad = 0.0;
    if ((rc = vec_dot(ctx, d, ad, n, &dad))) return rc;
    if (dad == 0.0) {
      if (last_step) *last_step = it;
      if (last_value) *last_value = res;
      return cg_status(3, it, res);
    }
    const double alpha = gh / dad;
    if ((rc = vec_axpy(ctx, x->d, 0.0, alpha, d, n, 0))) return rc;
    if ((rc = vec_axpy(ctx, g, 0.0, alpha, ad, n, 0))) return rc;
    if ((rc = vec_dot(ctx, g, g, n, &gg))) return rc;
    res = std::sqrt(gg);
    if (history && it < history_len) history[it] = res;
    if ((conv = control_check(control, it, max_its, res, tol)) != 0) break;
    if ((rc = vcycle(mg, top, mg->h, mg->g))) return rc;
    if (mg->profile) mg->n_vcycles++;
    const double gh_old = gh;
    if ((rc = vec_dot(ctx, g, mg->h->d, n, &gh))) return rc;
    if ((rc = vec_axpy(ctx, d, gh / gh_old, -1.0, mg->h->d, n, 2))) return rc;   // d = beta d - h
  }
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  if (last_step) *last_step = it;
  if (last_value) *last_value = res;
  return cg_status(conv, it, res);
  BP5_MG_GUARD_END
}

int bp5_mg_profile(bp5_mg_t mg, int enable) {
  BP5_REQUIRE(mg, "null argument");
  mg->profile = enable != 0;
  return BP5_OK;
}

int bp5_mg_profile_result(bp5_mg_t mg, double *ms, int64_t *n_vcycles) {
  BP5_REQUIRE(mg, "null argument");
  BP5_CUDA(cudaSetDevice(mg->ctx->device));
  int rc;
  if ((rc = prof_collect(mg))) return rc;
  if (ms) std::copy(mg->prof_ms.begin(), mg->prof_ms.end(), ms);
  if (n_vcycles) *n_vcycles = mg->n_vcycles;
  std::fill(mg->prof_ms.begin(), mg->prof_ms.end(), 0.0);
  mg->n_vcycles = 0;
  return BP5_OK;
}

}  // extern "C"
