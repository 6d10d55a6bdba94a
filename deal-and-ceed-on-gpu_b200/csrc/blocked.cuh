// Index map of the merged CG's blocked DoF layout (BlockedLayout, common.h).
#pragma once
#include "common.h"

namespace bp5 {

inline BlockedLayout make_blocked_layout(int p, const int *nc) {
  BlockedLayout L;
  L.p = p;
  for (int d = 0; d < 3; ++d) L.nc[d] = nc[d];
  L.nx = p * nc[0] + 1; L.ny = p * nc[1] + 1;
  L.ki = nc[2] * (p - 1); L.ji = nc[1] * (p - 1);
  const long long ii = (long long)nc[0] * (p - 1);
  L.sa = ii * L.ji * L.ki;
  L.sb = L.sa + (long long)(nc[2] + 1) * L.nx * L.ny;
  L.sc = L.sb + (long long)(nc[1] + 1) * L.ki * L.nx;
  L.n = L.sc + (long long)(nc[0] + 1) * L.ki * L.ji;
  return L;
}

// position of lattice point (i, j, k) of the block in the blocked layout
__host__ __device__ inline long long blocked_index(const BlockedLayout &L, int i, int j, int k) {
  const int p = L.p;
  const int ci = i / p, cj = j / p, ck = k / p;
  const int ri = i - ci * p, rj = j - cj * p, rk = k - ck * p;
  if (rk == 0) return L.sa + ((long long)ck * L.ny + j) * L.nx + i;
  const long long kk = (long long)ck * (p - 1) + rk - 1;
  if (rj == 0) return L.sb + ((long long)cj * L.ki + kk) * L.nx + i;
  const long long jj = (long long)cj * (p - 1) + rj - 1;
  if (ri == 0) return L.sc + ((long long)ci * L.ki + kk) * L.ji + jj;
  const long long cell = ((long long)ck * L.nc[1] + cj) * L.nc[0] + ci;
  return ((cell * (p - 1) + rk - 1) * (p - 1) + rj - 1) * (p - 1) + ri - 1;
}

}  // namespace bp5
