// BLAS-1 on the owned range of a distributed vector: the operations
// SolverCGFullMerge and the driver call on
// LinearAlgebra::distributed::Vector<double, MemorySpace::CUDA> [UPSTREAM]
// (bp5/solver.h:375-382,511 ; bp5/step-64.cu:445,449,467).
// Reductions are deterministic: fixed grid, per-block partials, one block sums
// them in a fixed order.
#include "blocked.cuh"

namespace bp5 {

constexpr int kRedBlocks = 592;   // 4 per SM on a 148-SM part
constexpr int kRedThreads = 256;

__global__ void fill_kernel(double *__restrict__ d, long long n, double v) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    d[i] = v;
}

// mode 0: y += a x ; 1: y = a x ; 2: y = s y + a x ; 3: y = y .* x
template <int MODE>
__global__ void axpy_kernel(double *__restrict__ y, double s, double a, const double *__restrict__ x, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    if (MODE == 0) y[i] += a * x[i];
    else if (MODE == 1) y[i] = a * x[i];
    else if (MODE == 2) y[i] = s * y[i] + a * x[i];
    else y[i] *= x[i];
  }
}

// the merged CG's layout change at the start and the end of a solve, one pass each
template <bool TO_BLOCKED>
__global__ void blocked_permute_kernel(BlockedLayout L, double *__restrict__ dst, const double *__restrict__ src,
                                       double scale) {
  const long long plane = (long long)L.nx * L.ny;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < L.n; t += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(t / plane);
    const int j = (int)((t - k * plane) / L.nx);
    const int i = (int)(t - k * plane - (long long)j * L.nx);
    const long long bi = blocked_index(L, i, j, k);
    if (TO_BLOCKED) dst[bi] = scale * src[t];
    else dst[t] = scale * src[bi];
  }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ double block_sum(double v, double *sh) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) sh[w] = v;
  __syncthreads();
  double r = 0.0;
  if (w == 0) {
    r = lane < (blockDim.x >> 5) ? sh[lane] : 0.0;
    r = warp_sum(r);
  }
  __syncthreads();
  return r;   // valid in warp 0
}

__global__ void dot_partial_kernel(const double *__restrict__ x, const double *__restrict__ y, long long n,
                                   double *__restrict__ partial) {
  __shared__ double sh[32];
  double s = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    s += x[i] * y[i];
  s = block_sum(s, sh);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void sum_partials_kernel(const double *__restrict__ partial, int n, double *__restrict__ out) {
  __shared__ double sh[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += partial[i];
  s = block_sum(s, sh);
  if (threadIdx.x == 0) *out = s;
}

__global__ void nonzero_kernel(const double *__restrict__ x, long long n, int *__restrict__ flag) {
  bool nz = false;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    nz |= (x[i] != 0.0);
  if (__syncthreads_or(nz) && threadIdx.x == 0) *flag = 1;
}

static unsigned grid_for(long long n, int threads, int cap) {
  long long g = (n + threads - 1) / threads;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (unsigned)g;
}

int vec_fill(bp5_context_t ctx, double *d, int64_t n, double v) {
  if (n == 0) return BP5_OK;
  if (v == 0.0) {
    BP5_CUDA(cudaMemsetAsync(d, 0, sizeof(double) * n, ctx->stream));
    return BP5_OK;
  }
  fill_kernel<<<grid_for(n, 256, 148 * 16), 256, 0, ctx->stream>>>(d, n, v);
  BP5_CHECK_LAUNCH();
  ctx->launches++;
  return BP5_OK;
}

int vec_axpy(bp5_context_t ctx, double *y, double s, double a, const double *x, int64_t n, int mode) {
  if (n == 0) return BP5_OK;
  const unsigned g = grid_for(n, 256, 148 * 16);
  if (mode == 0) axpy_kernel<0><<<g, 256, 0, ctx->stream>>>(y, s, a, x, n);
  else if (mode == 1) axpy_kernel<1><<<g, 256, 0, ctx->stream>>>(y, s, a, x, n);
  else if (mode == 2) axpy_kernel<2><<<g, 256, 0, ctx->stream>>>(y, s, a, x, n);
  else axpy_kernel<3><<<g, 256, 0, ctx->stream>>>(y, s, a, x, n);
  BP5_CHECK_LAUNCH();
  ctx->launches++;
  return BP5_OK;
}

int vec_blocked_permute(bp5_context_t ctx, const BlockedLayout &L, double *dst, const double *src, double scale,
                        bool to_blocked) {
  if (L.n == 0) return BP5_OK;
  const unsigned g = grid_for(L.n, 256, 148 * 16);
  if (to_blocked) blocked_permute_kernel<true><<<g, 256, 0, ctx->stream>>>(L, dst, src, scale);
  else blocked_permute_kernel<false><<<g, 256, 0, ctx->stream>>>(L, dst, src, scale);
  BP5_CHECK_LAUNCH();
  ctx->launches++;
  return BP5_OK;
}

// scratch layout: [0, kRedBlocks) partials, [kRedBlocks] result
int vec_dot(bp5_context_t ctx, const double *x, const double *y, int64_t n, double *out) {
  dot_partial_kernel<<<kRedBlocks, kRedThreads, 0, ctx->stream>>>(x, y, n, ctx->scratch);
  BP5_CHECK_LAUNCH();
  sum_partials_kernel<<<1, 256, 0, ctx->stream>>>(ctx->scratch, kRedBlocks, ctx->scratch + kRedBlocks);
  BP5_CHECK_LAUNCH();
  ctx->launches += 2;
  BP5_CUDA(cudaMemcpyAsync(ctx->scratch_host, ctx->scratch + kRedBlocks, sizeof(double), cudaMemcpyDeviceToHost,
                           ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  *out = ctx->scratch_host[0];
  return BP5_OK;
}

int vec_all_zero(bp5_context_t ctx, const double *x, int64_t n, int *out) {
  int *flag = reinterpret_cast<int *>(ctx->scratch + kRedBlocks + 1);
  BP5_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), ctx->stream));
  if (n > 0) {
    nonzero_kernel<<<grid_for(n, 256, 148 * 8), 256, 0, ctx->stream>>>(x, n, flag);
    BP5_CHECK_LAUNCH();
    ctx->launches++;
  }
  int *hflag = reinterpret_cast<int *>(ctx->scratch_host + 1);
  BP5_CUDA(cudaMemcpyAsync(hflag, flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  *out = (*hflag == 0);
  return BP5_OK;
}

}  // namespace bp5
