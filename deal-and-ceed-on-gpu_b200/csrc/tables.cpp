// 1D quadrature rules and shape tables of FE_Q(p) (host side).
// Replaces what the reference gets from deal.II: FE_Q<dim>(fe_degree)
// (bp5/step-64.cu:312,334), QGauss<1>(p+1) / QGaussLobatto<1>(p+1)
// (bp5/step-64.cu:243-247) and the shape_values / shape_gradients /
// co_shape_gradients that CUDAWrappers::MatrixFree::reinit copies to constant
// memory [UPSTREAM].
#include <cmath>
#include <cstring>

#include "common.h"

namespace bp5 {

namespace {
// Legendre polynomial L_m and its first derivative at z in (-1,1), carried
// together through Bonnet's recurrence.
struct Leg { long double v, d; };
Leg legendre_pair(int m, long double z) {
  long double v0 = 1.0L, v1 = z, d0 = 0.0L, d1 = 1.0L;
  if (m == 0) return {v0, d0};
  for (int k = 1; k < m; ++k) {
    const long double v2 = ((2 * k + 1) * z * v1 - k * v0) / (k + 1);
    const long double d2 = d0 + (2 * k + 1) * v1;   // L'_{k+1} = L'_{k-1} + (2k+1) L_k
    v0 = v1; v1 = v2; d0 = d1; d1 = d2;
  }
  return {v1, d1};
}
}  // namespace

void gauss_rule01(int n, double *x, double *w) {
  const long double pi = 3.14159265358979323846264338327950288L;
  for (int i = 0; i < (n + 1) / 2; ++i) {
    long double z = -cosl(pi * (4 * i + 3) / (4 * n + 2));   // Tricomi-like start
    for (int it = 0; it < 60; ++it) {
      const Leg l = legendre_pair(n, z);
      const long double step = l.v / l.d;
      z -= step;
      if (fabsl(step) < 1e-19L) break;
    }
    const Leg l = legendre_pair(n, z);
    const long double wt = 2.0L / ((1.0L - z * z) * l.d * l.d);
    x[i] = (double)(0.5L * (1.0L + z));
    x[n - 1 - i] = (double)(0.5L * (1.0L - z));
    w[i] = w[n - 1 - i] = (double)(0.5L * wt);
  }
  if (n % 2) x[n / 2] = 0.5;
}

void lobatto_rule01(int n, double *x, double *w) {
  const long double pi = 3.14159265358979323846264338327950288L;
  const int m = n - 1;   // nodes: +-1 and the roots of L_m'
  for (int i = 0; i < (n + 1) / 2; ++i) {
    long double z;
    if (i == 0)
      z = -1.0L;
    else {
      z = -cosl(pi * i / m);
      for (int it = 0; it < 60; ++it) {
        const Leg l = legendre_pair(m, z);
        // L_m'' from (1-z^2) L'' = 2 z L' - m(m+1) L
        const long double dd = (2.0L * z * l.d - (long double)m * (m + 1) * l.v) / (1.0L - z * z);
        const long double step = l.d / dd;
        z -= step;
        if (fabsl(step) < 1e-19L) break;
      }
    }
    const Leg l = legendre_pair(m, z);
    const long double wt = 2.0L / ((long double)m * (m + 1) * l.v * l.v);
    x[i] = (double)(0.5L * (1.0L + z));
    x[n - 1 - i] = (double)(0.5L * (1.0L - z));
    w[i] = w[n - 1 - i] = (double)(0.5L * wt);
  }
  if (n % 2) x[n / 2] = 0.5;
}

// Lagrange basis through `nodes`, value and derivative at x (barycentric-free
// product form; n <= 9 so conditioning is a non-issue).
void lagrange_eval(int n, const double *nodes, double x, double *val, double *der) {
  for (int a = 0; a < n; ++a) {
    long double denom = 1.0L;
    for (int b = 0; b < n; ++b)
      if (b != a) denom *= (long double)nodes[a] - nodes[b];
    long double v = 1.0L, dsum = 0.0L;
    for (int b = 0; b < n; ++b)
      if (b != a) v *= (long double)x - nodes[b];
    for (int c = 0; c < n; ++c) {
      if (c == a) continue;
      long double t = 1.0L;
      for (int b = 0; b < n; ++b)
        if (b != a && b != c) t *= (long double)x - nodes[b];
      dsum += t;
    }
    val[a] = (double)(v / denom);
    der[a] = (double)(dsum / denom);
  }
}

// 1D parent-to-child interpolation: out[s][a * n + b] = l_b((s + xi_a) / 2), the value of the parent's basis
// function b at node a of child s.  Hanging-node constraints and the multigrid transfer both use it.
void parent_child_interp(const Tables1D &t, double (*out)[kMaxN * kMaxN]) {
  const int n = t.n;
  for (int s = 0; s < 2; ++s)
    for (int a = 0; a < n; ++a) {
      double val[kMaxN], der[kMaxN];
      lagrange_eval(n, t.xi, 0.5 * (s + t.xi[a]), val, der);
      for (int b = 0; b < n; ++b) out[s][a * n + b] = val[b];
    }
}

void make_tables(int degree, int quadrature, Tables1D &t) {
  std::memset(&t, 0, sizeof(t));
  const int n = degree + 1;
  t.n = n;
  double scratch[kMaxN];
  lobatto_rule01(n, t.xi, scratch);
  if (quadrature == BP5_QUAD_GLL)
    lobatto_rule01(n, t.xq, t.wq);
  else
    gauss_rule01(n, t.xq, t.wq);
  double val[kMaxN], der[kMaxN];
  for (int q = 0; q < n; ++q) {
    lagrange_eval(n, t.xi, t.xq[q], val, der);
    for (int i = 0; i < n; ++i) {
      t.B[q * n + i] = (quadrature == BP5_QUAD_GLL) ? (q == i ? 1.0 : 0.0) : val[i];
      t.Dg[q * n + i] = der[i];
    }
    lagrange_eval(n, t.xq, t.xq[q], val, der);
    for (int r = 0; r < n; ++r) t.Dt[q * n + r] = der[r];
  }
}

}  // namespace bp5
