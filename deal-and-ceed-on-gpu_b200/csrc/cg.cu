// Conjugate gradients around the operator: SolverCGFullMerge::solve
// (bp5/solver.h:343-542) and dealii::SolverCG::solve as the driver uses it
// (bp5/step-64.cu:446-453) [UPSTREAM].
//
// What changed relative to the reference, and why (DESIGN.md section 4):
//  * alpha, beta, the residual and the stopping decision live in a small device
//    struct; the update kernels read them from memory.  The reference copies
//    seven doubles to the host with a blocking cudaMemcpy and runs
//    MPI_Allreduce every iteration (solver.h:489-494); here nothing crosses
//    PCIe inside the loop, the host only polls an "are we done" word every few
//    iterations, asynchronously.
//  * the seven dot products (update_b, solver.h:142-311) are reduced with warp
//    shuffles and per-block partials summed in a fixed order by the last block
//    to arrive (deterministic; the reference's shared-memory tree relies on
//    warp-synchronous execution, unsafe since sm_70), and the same block then
//    evaluates the scalar recurrences of solver.h:497-533.
//  * after convergence every kernel of the iteration turns into a no-op, so an
//    asynchronous host never changes the result or last_step().
//  * the two-step x update (update_a1, solver.h:106-140) is applied on odd
//    iterations only; as shipped (test at solver.h:425) it runs on every
//    iteration >= 3 and returns a wrong x (SURVEY.md finding 4).  Residual
//    history and iteration count are identical either way.
#include <algorithm>

#include "apply.cuh"
#include "cg_state.cuh"
#include "common.h"

namespace bp5 {

constexpr int kCgBlocks = 592;
constexpr int kCgThreads = 256;

constexpr int kUpdatePartialCap = 4096;     // >= grid of the update kernel (sm_count * 16)

// lays out CgBuffers (common.h) from `base`; returns the bytes they need
static size_t cg_layout(void *base, int hist_len, CgBuffers *b) {
  const size_t o_partials = 256;
  const size_t o_ph = o_partials + sizeof(double) * kCgBlocks * 7;
  const size_t o_rr = o_ph + sizeof(double) * (kApplyPartialCap + kConstrainedPartials);
  const size_t o_hist = o_rr + sizeof(double) * kUpdatePartialCap * 2;
  if (b) {
    char *c = reinterpret_cast<char *>(base);
    b->st = reinterpret_cast<CgState *>(c);
    b->partials = reinterpret_cast<double *>(c + o_partials);
    b->ph = reinterpret_cast<double *>(c + o_ph);
    b->rr = reinterpret_cast<double *>(c + o_rr);
    b->hist = hist_len > 0 ? reinterpret_cast<double *>(c + o_hist) : nullptr;
  }
  return o_hist + sizeof(double) * (hist_len > 0 ? hist_len : 1);
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// block-wide sums of K values; result valid in thread 0
template <int K>
__device__ __forceinline__ void block_sum_k(double (&v)[K], double *sh /*[K*32]*/) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int j = 0; j < K; ++j) v[j] = warp_sum_d(v[j]);
  if (lane == 0)
#pragma unroll
    for (int j = 0; j < K; ++j) sh[j * 32 + w] = v[j];
  __syncthreads();
  if (w == 0) {
#pragma unroll
    for (int j = 0; j < K; ++j) {
      double r = lane < nw ? sh[j * 32 + lane] : 0.0;
      v[j] = warp_sum_d(r);
    }
  }
  __syncthreads();
}

// ---------------------------------------------------------------- merged CG
// MODE 0: update_a0 (solver.h:48-72)  1: update_a<false> (:74-104)  3: update_a1 (:106-140)
// Fused here: r.r (and r.Dr) of the residual this kernel WRITES -- two of the seven sums of update_b
// (solver.h:142-311) -- as per-block partials rr[block][2], so the dots pass does not have to form them.
template <int MODE, bool DIAG>
__global__ void __launch_bounds__(256) cg_update_kernel(const CgState *__restrict__ st, double *__restrict__ p,
                                                        double *__restrict__ r, double *__restrict__ v,
                                                        double *__restrict__ x, const double *__restrict__ diag,
                                                        double *__restrict__ rr, long long n) {
  // "v = 0" (solver.h:69,101,137).  (Restricting it to the skeleton was measured slower: scattered
  // partial-sector writes, and L2 fills the sectors anyway.)
  if (st->state != 0) return;
  __shared__ double sh[2 * 32];
  const double alpha = st->alpha, beta = st->beta;
  double apa = 0.0, aob = 0.0;
  if (MODE == 3) { aob = st->alpha_old / st->beta_old; apa = alpha + aob; }
  double s[2] = {0.0, 0.0};
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double dg = DIAG ? diag[i] : 1.0;
    double r_new;
    if (MODE == 0) {
      r_new = r[i];
      p[i] = -dg * r_new;
    } else {
      const double r_old = r[i];
      r_new = r_old + alpha * v[i];
      const double p_old = p[i];
      if (MODE == 3) x[i] += apa * p_old + aob * dg * r_old;
      r[i] = r_new;
      p[i] = beta * p_old - dg * r_new;
    }
    v[i] = 0.0;
    s[0] += r_new * r_new;
    if (DIAG) s[1] += r_new * dg * r_new;
  }
  block_sum_k<2>(s, sh);
  if (threadIdx.x == 0) { rr[2 * blockIdx.x] = s[0]; rr[2 * blockIdx.x + 1] = s[1]; }
}

// partitioned meshes: the sums come back from an allreduce over the blocks
__global__ void cg_scalars_kernel(CgState *st, const double *__restrict__ sums, double *history) {
  if (st->state != 0 || threadIdx.x != 0 || blockIdx.x != 0) return;
  double rr[7];
#pragma unroll
  for (int j = 0; j < 7; ++j) rr[j] = sums[j];
  cg_scalar_step(st, rr, history);
}

// FUSE: the last block also runs the scalar recurrences (single block of the mesh);
// otherwise it writes the seven local sums to sums_out for the caller's allreduce.
// LEAN: p.v comes from the cell kernel (n_ph per-CTA partials in ph: cells + Dirichlet correction) and
// r.r / r.Dr from the update kernel (n_rr per-block partials in rr): only r and v are read here.
template <bool DIAG, bool FUSE, bool LEAN>
__global__ void __launch_bounds__(kCgThreads) cg_dots_kernel(CgState *st, const double *__restrict__ p,
                                                             const double *__restrict__ r,
                                                             const double *__restrict__ v,
                                                             const double *__restrict__ diag, long long n,
                                                             double *partials, double *history, double *sums_out,
                                                             const double *ph, int n_ph, const double *rr, int n_rr) {
  if (st->state != 0) return;
  __shared__ double sh[7 * 32];
  __shared__ bool is_last;
  constexpr int K = DIAG ? 7 : 4;
  double s[K];
#pragma unroll
  for (int j = 0; j < K; ++j) s[j] = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double rs = r[i], vs = v[i];
    s[1] += vs * vs; s[2] += rs * vs;
    if (!LEAN) { s[0] += p[i] * vs; s[3] += rs * rs; }
    if (DIAG) {
      const double ds = diag[i], dv = ds * vs;
      s[4] += rs * dv; s[5] += vs * dv;
      if (!LEAN) s[6] += rs * ds * rs;
    }
  }
  block_sum_k<K>(s, sh);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int j = 0; j < K; ++j) partials[blockIdx.x * 7 + j] = s[j];
    __threadfence();
    const unsigned t = atomicAdd(&st->ticket, 1u);
    is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // last block: fixed-order sum of the partials, then the scalar recurrences
#pragma unroll
  for (int j = 0; j < K; ++j) s[j] = 0.0;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x)
#pragma unroll
    for (int j = 0; j < K; ++j) s[j] += __ldcg(&partials[b * 7 + j]);
  if (LEAN) {
    s[0] = 0.0; s[3] = 0.0;
    if (DIAG) s[6] = 0.0;
    for (int b = threadIdx.x; b < n_ph; b += blockDim.x) s[0] += __ldcg(&ph[b]);
    for (int b = threadIdx.x; b < n_rr; b += blockDim.x) {
      s[3] += __ldcg(&rr[2 * b]);
      if (DIAG) s[6] += __ldcg(&rr[2 * b + 1]);
    }
  }
  block_sum_k<K>(s, sh);
  if (threadIdx.x == 0) {
    double q[7];
#pragma unroll
    for (int j = 0; j < K; ++j) q[j] = s[j];
    if (!DIAG) { q[4] = q[2]; q[5] = q[1]; q[6] = q[3]; }
    st->ticket = 0;
    if (FUSE) cg_scalar_step(st, q, history);
    else
#pragma unroll
      for (int j = 0; j < 7; ++j) sums_out[j] = q[j];
  }
}

// x update owed at termination (solver.h:509-526)
template <bool DIAG>
__global__ void cg_finish_kernel(const CgState *__restrict__ st, double *__restrict__ x,
                                 const double *__restrict__ d, const double *__restrict__ g,
                                 const double *__restrict__ diag, long long n) {
  if (st->state == 0 || st->state == 3 || st->it == 0) return;
  const double alpha = st->alpha;
  const bool odd = (st->it % 2) == 1;
  double apa = 0.0, aob = 0.0;
  if (!odd) { aob = st->alpha_old / st->beta_old; apa = alpha + aob; }
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    if (odd) x[i] += alpha * d[i];
    else x[i] += apa * d[i] + aob * (DIAG ? diag[i] : 1.0) * g[i];
  }
}

// -------------------------------------------------------------- standard CG
// d = -D g, h = D g
template <bool DIAG>
__global__ void std_init_kernel(double *__restrict__ d, double *__restrict__ h, const double *__restrict__ g,
                                const double *__restrict__ diag, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double hv = (DIAG ? diag[i] : 1.0) * g[i];
    h[i] = hv; d[i] = -hv;
  }
}

// alpha = gh / (d.h), d.h summed from the cell kernel's per-CTA partials of d.(A d) (+ Dirichlet correction):
// one block, fixed order
__global__ void __launch_bounds__(kCgThreads) std_alpha_kernel(CgState *st, const double *__restrict__ ph, int n_ph) {
  if (st->state != 0) return;
  __shared__ double sh[32];
  double s[1] = {0.0};
  for (int b = threadIdx.x; b < n_ph; b += blockDim.x) s[0] += ph[b];
  block_sum_k<1>(s, sh);
  if (threadIdx.x == 0) {
    if (s[0] == 0.0) { st->state = 3; return; }
    st->alpha = st->gh / s[0];
  }
}

// x += alpha d ; g += alpha h ; res = |g| ; check ; beta = (g.Dg)/gh ; gh = g.Dg
template <bool DIAG>
__global__ void __launch_bounds__(kCgThreads) std_xg_kernel(CgState *st, double *__restrict__ x,
                                                            double *__restrict__ g, const double *__restrict__ d,
                                                            const double *__restrict__ h,
                                                            const double *__restrict__ diag, long long n,
                                                            double *partials, double *history) {
  if (st->state != 0) return;
  __shared__ double sh[2 * 32];
  __shared__ bool is_last;
  const double alpha = st->alpha;
  double s[2] = {0.0, 0.0};
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    x[i] += alpha * d[i];
    const double gn = g[i] + alpha * h[i];
    g[i] = gn;
    s[0] += gn * gn;
    s[1] += gn * (DIAG ? diag[i] : 1.0) * gn;
  }
  block_sum_k<2>(s, sh);
  if (threadIdx.x == 0) {
    partials[blockIdx.x * 7] = s[0];
    partials[blockIdx.x * 7 + 1] = s[1];
    __threadfence();
    is_last = (atomicAdd(&st->ticket, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  s[0] = s[1] = 0.0;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
    s[0] += __ldcg(&partials[b * 7]);
    s[1] += __ldcg(&partials[b * 7 + 1]);
  }
  block_sum_k<2>(s, sh);
  if (threadIdx.x == 0) {
    st->ticket = 0;
    const int it = st->it + 1;
    st->it = it;
    const double res = sqrt(s[0]);
    st->res = res;
    if (history && it < st->history_len) history[it] = res;
    const int conv = control_check(st->control, it, st->max_its, res, st->tol);
    if (conv != 0) { st->state = conv; return; }
    st->beta = s[1] / st->gh;
    st->gh = s[1];
  }
}

// d = beta d - D g
template <bool DIAG>
__global__ void std_d_kernel(const CgState *__restrict__ st, double *__restrict__ d, const double *__restrict__ g,
                             const double *__restrict__ diag, long long n) {
  if (st->state != 0) return;
  const double beta = st->beta;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    d[i] = beta * d[i] - (DIAG ? diag[i] : 1.0) * g[i];
}

static unsigned stream_grid(long long n, int sm_count) {
  long long g = (n + 255) / 256;
  const long long cap = (long long)sm_count * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (unsigned)g;
}

int cg_buffers(bp5_operator_t op, int hist_len, CgBuffers *cb) {
  int rc;
  // temporary vectors g, d, h (VectorMemory pool in the reference, solver.h:355-371); kept with the operator
  if (!op->g) {
    if ((rc = bp5_vector_create(op->ctx, op->n_owned, op->n_ghost, &op->g))) return rc;
    if ((rc = bp5_vector_create(op->ctx, op->n_owned, op->n_ghost, &op->d))) return rc;
    if ((rc = bp5_vector_create(op->ctx, op->n_owned, op->n_ghost, &op->h))) return rc;
  }
  const size_t need = cg_layout(nullptr, hist_len, nullptr);
  if (!op->cg_scalars || op->cg_scalars_bytes < need) {
    if (op->cg_scalars) cudaFree(op->cg_scalars);
    op->cg_scalars = nullptr;
    BP5_CUDA(cudaMalloc(&op->cg_scalars, need));
    op->cg_scalars_bytes = need;
  }
  if (cb) cg_layout(op->cg_scalars, hist_len, cb);
  return BP5_OK;
}

int cg_status(int state, int it, double res) {
  if (state == 3) { set_error("ExcDivideByZero: d.Ad == 0 at iteration %d", it); return BP5_ERR_DIVIDE_BY_ZERO; }
  if (state == 2) { set_error("NoConvergence: step %d, residual %.17g", it, res); return BP5_ERR_NO_CONVERGENCE; }
  if (state != 1) { set_error("CG ended in unexpected state %d", state); return BP5_ERR_INVALID; }
  return BP5_OK;
}

// The pieces of one merged-CG iteration, on the context's stream.  cg_solve() (single block), the stepwise API
// (partitioned meshes, the caller's transport in between) and cg_solve_peer() all run these; everything they call
// only enqueues work, so cg_solve() and cg_solve_peer() can capture them into a CUDA graph.
//
// 1) update region (solver.h:413-448) of iteration `cur` (1-based), with the parity-correct x update, plus r.r and
//    r.Dr of the new residual as per-block partials in cb.rr.  The kernel zeroes h; its ghost entries receive the
//    contributions for the neighbouring owners, so they start at zero too.
template <int MODE>
static void launch_update(unsigned grid, cudaStream_t s, const CgBuffers &cb, double *p, double *r, double *v,
                          double *x, const double *diag, long long n) {
  if (diag) cg_update_kernel<MODE, true><<<grid, 256, 0, s>>>(cb.st, p, r, v, x, diag, cb.rr, n);
  else cg_update_kernel<MODE, false><<<grid, 256, 0, s>>>(cb.st, p, r, v, x, diag, cb.rr, n);
}

static int enqueue_update(bp5_operator_t op, const CgBuffers &cb, int cur, double *x, const double *diag) {
  const long long n = op->n_owned;
  const unsigned grid = stream_grid(n, op->ctx->sm_count);
  BP5_REQUIRE(grid <= (unsigned)kUpdatePartialCap, "update grid exceeds the partial-sum buffer");
  cudaStream_t s = op->ctx->stream;
  double *g = op->g->d, *d = op->d->d, *h = op->h->d;
  if (cur == 1) launch_update<0>(grid, s, cb, d, g, h, x, diag, n);
  else if (cur % 2 == 0) launch_update<1>(grid, s, cb, d, g, h, x, diag, n);
  else launch_update<3>(grid, s, cb, d, g, h, x, diag, n);
  BP5_CHECK_LAUNCH();
  op->ctx->launches++;
  if (op->n_ghost) BP5_CUDA(cudaMemsetAsync(h + n, 0, sizeof(double) * op->n_ghost, s));
  return BP5_OK;
}

// 2) h = A d: apply_cell_loop(op, h, d, true, cb.ph) with do_zero_out = false (solver.h:475; h's skeleton is zeroed by
//    the update kernel, its cell-interior entries are overwritten by the cell kernel) leaves d.h as per-CTA partials.
// 3) Dirichlet copy h_c = d_c, with its correction of d.h after the cell loop's n_ph partials.
static int enqueue_constrained(bp5_operator_t op, const CgBuffers &cb, int n_ph) {
  if (op->n_constrained == 0) return BP5_OK;
  return apply_copy_constrained_dot(op, op->h->d, op->d->d, cb.ph + n_ph);
}

// partials of d.h once the Dirichlet copy has followed a cell loop that left n_ph
static int ph_count(bp5_operator_t op, int n_ph) { return n_ph + (op->n_constrained > 0 ? kConstrainedPartials : 0); }

// 4) the remaining dots (h.h, r.h, r.Dh, h.Dh) over r = g, v = h, p = d; FUSE: and the scalars (solver.h:478-533),
//    otherwise the seven local sums go to sums_out.  lean: d.h from n_ph partials in cb.ph and r.r, r.Dr from n_rr in
//    cb.rr.
template <bool FUSE>
static int enqueue_dots(bp5_operator_t op, const CgBuffers &cb, const double *diag, bool lean, double *sums_out,
                        int n_ph, int n_rr) {
  cudaStream_t s = op->ctx->stream;
  const double *p = op->d->d, *r = op->g->d, *v = op->h->d;
  const long long n = op->n_owned;
#define BP5_DOTS(D, L)                                                                                          \
  cg_dots_kernel<D, FUSE, L><<<kCgBlocks, kCgThreads, 0, s>>>(cb.st, p, r, v, diag, n, cb.partials, cb.hist, sums_out, \
                                                            cb.ph, n_ph, cb.rr, n_rr)
  if (diag) { if (lean) BP5_DOTS(true, true); else BP5_DOTS(true, false); }
  else { if (lean) BP5_DOTS(false, true); else BP5_DOTS(false, false); }
#undef BP5_DOTS
  BP5_CHECK_LAUNCH();
  op->ctx->launches++;
  return BP5_OK;
}

// x update owed at termination (solver.h:509-526)
static int enqueue_finish(bp5_operator_t op, const CgState *st, double *x, const double *diag) {
  const long long n = op->n_owned;
  const unsigned grid = stream_grid(n, op->ctx->sm_count);
  cudaStream_t s = op->ctx->stream;
  if (diag) cg_finish_kernel<true><<<grid, 256, 0, s>>>(st, x, op->d->d, op->g->d, diag, n);
  else cg_finish_kernel<false><<<grid, 256, 0, s>>>(st, x, op->d->d, op->g->d, diag, n);
  BP5_CHECK_LAUNCH();
  op->ctx->launches++;
  return BP5_OK;
}

// Iteration loop shared by cg_solve() and cg_solve_peer().  `enqueue(cur)` puts iteration `cur` (1-based) on the
// stream.  The first kWarm iterations are enqueued directly (they also trigger the one-time kernel attribute
// set-up); after that one batch of kBatch iterations is captured into a CUDA graph and replayed, which removes
// most of the launch latency that dominates small blocks (everything an iteration needs -- alpha, beta, epochs,
// the "converged, do nothing" word -- lives in device memory, so the replay needs no new arguments).  After each
// batch the state word of the batch before last is polled, so the GPU never waits for the host; iterations
// enqueued past convergence or past max_its are no-ops.
template <typename Enqueue>
static int run_iterations(bp5_operator_t op, CgState *st, int max_its, Enqueue enqueue) {
  bp5_context_t ctx = op->ctx;
  cudaStream_t s = ctx->stream;
  constexpr int kBatch = 8, kWarm = 3;                  // kWarm odd, kBatch even: a batch starts on an even iteration
  const bool use_graph = !op->profile && max_its >= kWarm + 2 * kBatch && getenv("BP5_NO_GRAPH") == nullptr;
  volatile int *poll_host = reinterpret_cast<volatile int *>(ctx->scratch_host + 8);   // two slots
  cudaEvent_t ev[2] = {nullptr, nullptr};
  BP5_CUDA(cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming));
  BP5_CUDA(cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming));
  poll_host[0] = poll_host[1] = 0;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t gexec = nullptr;
  int64_t launches_per_graph = 0;
  int it = 0, nbatch = 0, rc = BP5_OK;
  bool done = false;
  while (!done && it < max_its && rc == BP5_OK) {
    if (use_graph && it >= kWarm) {
      if (!gexec) {
        const int64_t l0 = ctx->launches;
        if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { rc = BP5_ERR_CUDA; break; }
        for (int k = 0; k < kBatch && rc == BP5_OK; ++k) rc = enqueue(it + 1 + k);
        const cudaError_t ee = cudaStreamEndCapture(s, &graph);
        if (rc != BP5_OK) break;
        if (ee != cudaSuccess || cudaGraphInstantiate(&gexec, graph, 0) != cudaSuccess) {
          set_error("CUDA graph capture of the CG batch failed: %s", cudaGetErrorString(cudaGetLastError()));
          rc = BP5_ERR_CUDA;
          break;
        }
        launches_per_graph = ctx->launches - l0;
        ctx->launches = l0;
      }
      if (cudaGraphLaunch(gexec, s) != cudaSuccess) { rc = BP5_ERR_CUDA; break; }
      ctx->launches += launches_per_graph;
      it += kBatch;
    } else {
      const int upto = std::min(max_its, it + (it < kWarm ? kWarm - it : kBatch));
      for (; it < upto && rc == BP5_OK; ++it) rc = enqueue(it + 1);
    }
    if (rc != BP5_OK) break;
    const int slot = nbatch & 1;
    if (cudaMemcpyAsync((void *)&poll_host[slot], &st->state, sizeof(int), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaEventRecord(ev[slot], s) != cudaSuccess) { rc = BP5_ERR_CUDA; break; }
    if (nbatch >= 1) {
      if (cudaEventSynchronize(ev[slot ^ 1]) != cudaSuccess) { rc = BP5_ERR_CUDA; break; }
      if (poll_host[slot ^ 1] != 0) done = true;
    }
    ++nbatch;
  }
  if (rc == BP5_ERR_CUDA && get_error()[0] == 0) set_error("CUDA error in the CG loop: %s", cudaGetErrorString(cudaGetLastError()));
  if (gexec) {
    cudaStreamSynchronize(s);
    cudaGraphExecDestroy(gexec);
  }
  if (graph) cudaGraphDestroy(graph);
  cudaEventDestroy(ev[0]);
  cudaEventDestroy(ev[1]);
  return rc;
}

// End of cg_solve() / cg_solve_peer() after run_iterations() returned rc: the owed x update (x == nullptr: none, as
// in the standard CG), the final state, history[1..], last_step / last_value and the return code.  peer: the
// transport's error word is checked before the state is decoded.
static int finish_solve(bp5_operator_t op, const CgBuffers &cb, int rc, double *x, const double *diag, bool peer,
                        double *history, int hist_len, int *last_step, double *last_value) {
  cudaStream_t s = op->ctx->stream;
  op->skip_flag = nullptr;
  if (rc == BP5_OK && x) rc = enqueue_finish(op, cb.st, x, diag);
  CgState fin{};
  cudaError_t e1 = cudaMemcpyAsync(&fin, cb.st, sizeof(CgState), cudaMemcpyDeviceToHost, s);
  cudaError_t e2 = cudaStreamSynchronize(s);
  if (rc != BP5_OK) return rc;
  if (e1 != cudaSuccess || e2 != cudaSuccess) {
    set_error("CG loop failed: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
    return BP5_ERR_CUDA;
  }
  BP5_CHECK_LAUNCH();
  if (peer && (rc = peer_check(op))) return rc;
  if (history && hist_len > 1) {
    const int cnt = std::min(hist_len, fin.it + 1) - 1;
    if (cnt > 0) BP5_CUDA(cudaMemcpy(history + 1, cb.hist + 1, sizeof(double) * cnt, cudaMemcpyDeviceToHost));
  }
  if (last_step) *last_step = fin.it;
  if (last_value) *last_value = fin.res;
  return cg_status(fin.state, fin.it, fin.res);
}

int cg_solve(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diagv, int variant, int control,
             double tol, int max_its, int *last_step, double *last_value, double *history, int history_len) {
  bp5_context_t ctx = op->ctx;
  cudaStream_t s = ctx->stream;
  const long long n = op->n_owned;
  BP5_REQUIRE(x->n_owned == n && b->n_owned == n, "vector size does not match the operator");
  BP5_REQUIRE(op->n_ghost == 0, "bp5_cg_solve handles a single block; partitioned meshes use the stepwise API");
  BP5_REQUIRE(max_its >= 0, "max_its must be >= 0");
  BP5_REQUIRE(variant == BP5_CG_MERGED || variant == BP5_CG_STANDARD, "unknown CG variant");
  const double *diag = diagv ? diagv->d : nullptr;
  const int hist_len = history ? history_len : 0;
  int rc;
  CgBuffers cb;
  if ((rc = cg_buffers(op, hist_len, &cb))) return rc;
  CgState *st = cb.st;
  double *g = op->g->d, *d = op->d->d, *h = op->h->d;

  // g = A x - b, or -b if x == 0 (solver.h:375-381)
  int x_zero = 0;
  if ((rc = vec_all_zero(ctx, x->d, n, &x_zero))) return rc;
  if (!x_zero) {
    if ((rc = apply_zero_skeleton(op, g))) return rc;
    if ((rc = apply_cell_loop(op, g, x->d, true))) return rc;
    if ((rc = apply_copy_constrained(op, g, x->d))) return rc;
    if ((rc = vec_axpy(ctx, g, 1.0, -1.0, b->d, n, 0))) return rc;
  } else if ((rc = vec_axpy(ctx, g, 0.0, -1.0, b->d, n, 1)))
    return rc;
  double gg = 0.0;
  if ((rc = vec_dot(ctx, g, g, n, &gg))) return rc;
  double res = std::sqrt(gg);
  if (history && history_len > 0) history[0] = res;

  const int conv = control_check(control, 0, max_its, res, tol);   // iteration_status(0, res_norm, x), solver.h:384
  if (conv != 0) {
    if (last_step) *last_step = 0;
    if (last_value) *last_value = res;
    return cg_status(conv, 0, res);
  }

  CgState init{};
  init.tol = tol; init.res = res; init.max_its = max_its; init.control = control; init.history_len = hist_len;
  const unsigned grid = stream_grid(n, ctx->sm_count);
  if (variant == BP5_CG_STANDARD) {
    if (diag) std_init_kernel<true><<<grid, 256, 0, s>>>(d, h, g, diag, n);
    else std_init_kernel<false><<<grid, 256, 0, s>>>(d, h, g, diag, n);
    BP5_CHECK_LAUNCH();
    ctx->launches++;
    double gh = 0.0;
    if ((rc = vec_dot(ctx, g, h, n, &gh))) return rc;
    init.gh = gh;
  }
  BP5_CUDA(cudaMemcpyAsync(st, &init, sizeof(CgState), cudaMemcpyHostToDevice, s));

  op->skip_flag = &st->state;
  auto enqueue = [&](int cur) -> int {
    int rc;
    if (variant == BP5_CG_MERGED) {   // the stepwise sequence, with the scalar recurrences fused into the dots kernel
      if ((rc = enqueue_update(op, cb, cur, x->d, diag))) return rc;
      if ((rc = apply_cell_loop(op, h, d, true, cb.ph))) return rc;
      if ((rc = enqueue_constrained(op, cb, op->apply_grid))) return rc;
      return enqueue_dots<true>(op, cb, diag, /*lean=*/true, nullptr, ph_count(op, op->apply_grid), (int)grid);
    }
    if ((rc = apply_zero_skeleton(op, h))) return rc;
    if ((rc = apply_cell_loop(op, h, d, true, cb.ph))) return rc;
    if ((rc = enqueue_constrained(op, cb, op->apply_grid))) return rc;
    std_alpha_kernel<<<1, kCgThreads, 0, s>>>(st, cb.ph, ph_count(op, op->apply_grid));   // alpha = gh / (d.h)
    if (diag) {
      std_xg_kernel<true><<<kCgBlocks, kCgThreads, 0, s>>>(st, x->d, g, d, h, diag, n, cb.partials, cb.hist);
      std_d_kernel<true><<<grid, 256, 0, s>>>(st, d, g, diag, n);
    } else {
      std_xg_kernel<false><<<kCgBlocks, kCgThreads, 0, s>>>(st, x->d, g, d, h, diag, n, cb.partials, cb.hist);
      std_d_kernel<false><<<grid, 256, 0, s>>>(st, d, g, diag, n);
    }
    ctx->launches += 3;
    return BP5_OK;
  };
  rc = run_iterations(op, st, max_its, enqueue);
  return finish_solve(op, cb, rc, variant == BP5_CG_MERGED ? x->d : nullptr, diag, /*peer=*/false, history, hist_len,
                      last_step, last_value);
}

// ------------------------------------------------------------------------
// Stepwise merged CG for partitioned meshes.  The host that owns the
// communicator interleaves: update -> [halo: update_ghost_values(d)] -> cell loop
// -> [halo: compress(add)(h)] -> Dirichlet copy -> local dots -> [allreduce of 7
// doubles, solver.h:493] -> scalars.  Nothing here synchronises except poll().
int cg_step_begin(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diag, int control, double tol,
                  int max_its, double res0, int history_len) {
  int rc;
  if ((rc = cg_buffers(op, history_len, &op->cg_buf))) return rc;
  op->cg_x = x; op->cg_diag = diag; op->cg_hist_len = history_len;
  const long long n = op->n_owned;
  // g = -b  (x == 0 on entry: g = A x - b, solver.h:375-381), ghosts zero
  BP5_CUDA(cudaMemsetAsync(op->g->d, 0, sizeof(double) * (n + op->n_ghost), op->ctx->stream));
  if ((rc = vec_axpy(op->ctx, op->g->d, 0.0, -1.0, b->d, n, 1))) return rc;
  CgState init{};
  init.tol = tol; init.res = res0; init.max_its = max_its; init.control = control; init.history_len = history_len;
  BP5_CUDA(cudaMemcpyAsync(op->cg_buf.st, &init, sizeof(CgState), cudaMemcpyHostToDevice, op->ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(op->ctx->stream));   // `init` lives on this stack frame
  op->skip_flag = &op->cg_buf.st->state;
  return BP5_OK;
}

int cg_step_update(bp5_operator_t op, int cur) {
  op->cg_ph_valid = false;       // set again by cg_step_apply_local; a foreign vmult leaves it false
  op->cg_update_grid = (int)stream_grid(op->n_owned, op->ctx->sm_count);
  return enqueue_update(op, op->cg_buf, cur, op->cg_x->d, op->cg_diag ? op->cg_diag->d : nullptr);
}

// 2) local cells' part of h = A d, with the fused d.h partials
int cg_step_apply_local(bp5_operator_t op) {
  const int rc = apply_cell_loop(op, op->h->d, op->d->d, true, op->cg_buf.ph);
  if (rc == BP5_OK) op->cg_ph_valid = true;
  return rc;
}

// Dirichlet copy after the halo sum; keeps the fused d.h consistent with h_c = d_c
int cg_step_constrained(bp5_operator_t op) {
  if (op->n_constrained == 0) return BP5_OK;
  if (!op->cg_ph_valid) return apply_copy_constrained(op, op->h->d, op->d->d);
  return enqueue_constrained(op, op->cg_buf, op->apply_grid);
}

int cg_step_local_dots(bp5_operator_t op, double *sums_dev) {
  const double *diag = op->cg_diag ? op->cg_diag->d : nullptr;
  // after a foreign vmult (user-written operator) there are no cell-kernel partials: read d as well
  const bool lean = op->cg_ph_valid;
  return enqueue_dots<false>(op, op->cg_buf, diag, lean, sums_dev, lean ? ph_count(op, op->apply_grid) : 0,
                             op->cg_update_grid);
}

int cg_step_scalars(bp5_operator_t op, const double *sums_dev) {
  cg_scalars_kernel<<<1, 32, 0, op->ctx->stream>>>(op->cg_buf.st, sums_dev, op->cg_buf.hist);
  BP5_CHECK_LAUNCH();
  op->ctx->launches++;
  return BP5_OK;
}

int cg_step_poll(bp5_operator_t op, int *state, int *it, double *res) {
  CgState fin{};
  BP5_CUDA(cudaMemcpyAsync(&fin, op->cg_buf.st, sizeof(CgState), cudaMemcpyDeviceToHost, op->ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(op->ctx->stream));
  if (state) *state = fin.state;
  if (it) *it = fin.it;
  if (res) *res = fin.res;
  return BP5_OK;
}

int cg_step_finish(bp5_operator_t op, double *history) {
  cudaStream_t s = op->ctx->stream;
  int rc;
  if ((rc = enqueue_finish(op, op->cg_buf.st, op->cg_x->d, op->cg_diag ? op->cg_diag->d : nullptr))) return rc;
  op->skip_flag = nullptr;
  if (history && op->cg_hist_len > 1)
    BP5_CUDA(cudaMemcpyAsync(history + 1, op->cg_buf.hist + 1, sizeof(double) * (op->cg_hist_len - 1),
                             cudaMemcpyDeviceToHost, s));
  BP5_CUDA(cudaStreamSynchronize(s));
  return BP5_OK;
}

// ------------------------------------------------------------------------
// Merged CG over a partitioned mesh with the peer-memory transport (peer.cu): the whole loop is
// enqueued from here, one rank per GPU, every rank the same sequence.  Per iteration:
//   update (r, p, x; h = 0; r.r partials) -> forward halo of d -> boundary cells -> reverse halo of h
//   -> interior cells (overlapping the reverse halo) -> add contributions -> Dirichlet copy
//   -> local dots -> all-rank sum through the mailboxes -> scalar recurrences.
// No NCCL / MPI call and no host synchronisation inside the loop; the host polls the state word of the
// batch before last like cg_solve().  The sums are added in rank order on every rank, so alpha, beta and
// the stopping decision are bitwise identical everywhere and all ranks stop in the same iteration.
int cg_solve_peer(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diagv, int control, double tol,
                  int max_its, int *last_step, double *last_value, double *history, int history_len) {
  BP5_REQUIRE(op->peer && op->peer_connected, "peer transport not connected (bp5_peer_export / bp5_peer_connect)");
  BP5_REQUIRE(max_its >= 0, "max_its must be >= 0");
  bp5_context_t ctx = op->ctx;
  cudaStream_t s = ctx->stream;
  const long long n = op->n_owned;
  const double *diag = diagv ? diagv->d : nullptr;
  const int hist_len = history ? history_len : 0;
  int rc;
  CgBuffers cb;
  if ((rc = cg_buffers(op, hist_len, &cb))) return rc;
  CgState *st = cb.st;
  double *g = op->g->d, *d = op->d->d, *h = op->h->d;
  double *sums = peer_scratch(op);            // [0,8) local, [8,16) global

  // g = -b (x == 0 on entry), ghosts zero; res0 = global |g|
  int x_zero = 0;
  if ((rc = vec_all_zero(ctx, x->d, n, &x_zero))) return rc;
  double flag[1] = {x_zero ? 0.0 : 1.0};
  if ((rc = peer_allreduce_host(op, flag, 1))) return rc;
  BP5_REQUIRE(flag[0] == 0.0, "bp5_peer_cg_solve needs x == 0 on entry");
  BP5_CUDA(cudaMemsetAsync(g, 0, sizeof(double) * (n + op->n_ghost), s));
  if ((rc = vec_axpy(ctx, g, 0.0, -1.0, b->d, n, 1))) return rc;
  double gg[1] = {0.0};
  if ((rc = vec_dot(ctx, g, g, n, &gg[0]))) return rc;
  if ((rc = peer_allreduce_host(op, gg, 1))) return rc;
  const double res0 = std::sqrt(gg[0]);
  if (history && history_len > 0) history[0] = res0;
  const int conv = control_check(control, 0, max_its, res0, tol);
  if (conv != 0) {
    if (last_step) *last_step = 0;
    if (last_value) *last_value = res0;
    return cg_status(conv, 0, res0);
  }
  CgState init{};
  init.tol = tol; init.res = res0; init.max_its = max_its; init.control = control; init.history_len = hist_len;
  BP5_CUDA(cudaMemcpyAsync(st, &init, sizeof(CgState), cudaMemcpyHostToDevice, s));
  BP5_CUDA(cudaStreamSynchronize(s));
  const unsigned grid = stream_grid(n, ctx->sm_count);

  op->skip_flag = &st->state;
  auto enqueue = [&](int cur) -> int {
    int rc;
    if ((rc = enqueue_update(op, cb, cur, x->d, diag))) return rc;
    // Both halves of the halo exchange hide behind cells that need no ghost data (MatrixFree's
    // overlap_communication_computation, bp5/step-64.cu:241): the upper faces of d leave for the neighbours, the
    // first half of the interior tiles runs, then the boundary tiles (they wait for the ghosts), the ghost
    // contributions leave, the second half of the interior runs, then the contributions that arrived are added.
    if ((rc = peer_forward(op, d, /*wait=*/false))) return rc;
    const long long n_int = op->n_tiles - op->n_boundary_tiles, half = op->n_boundary_tiles + n_int / 2;
    op->range_begin = op->n_boundary_tiles; op->range_end = half;
    rc = apply_cell_loop(op, h, d, true, cb.ph);
    op->range_begin = op->range_end = -1;
    if (rc) return rc;
    const int grid_a = op->apply_grid;
    if ((rc = peer_wait_forward(op))) return rc;
    if ((rc = apply_cell_loop(op, h, d, true, cb.ph + grid_a, 1))) return rc;
    const int grid_b = grid_a + op->apply_grid;
    if ((rc = peer_reverse(op, h))) return rc;
    op->range_begin = half; op->range_end = op->n_tiles;
    rc = apply_cell_loop(op, h, d, true, cb.ph + grid_b);
    op->range_begin = op->range_end = -1;
    if (rc) return rc;
    const int n_ph = grid_b + op->apply_grid;
    // boundary + interior partials + the Dirichlet correction share cb.ph: the next buffer (r.r partials) must
    // never be reached
    BP5_REQUIRE(ph_count(op, n_ph) <= kApplyPartialCap + kConstrainedPartials, "cell-kernel partial sums exceed their buffer");
    if ((rc = peer_wait_add(op, h))) return rc;
    if ((rc = enqueue_constrained(op, cb, n_ph))) return rc;
    if ((rc = enqueue_dots<false>(op, cb, diag, /*lean=*/true, sums, ph_count(op, n_ph), (int)grid))) return rc;
    // all-rank sum of the seven scalars; the same one-block kernel then runs the scalar recurrences
    return peer_allreduce(op, sums, sums + 8, 7, true, st, cb.hist);
  };
  rc = run_iterations(op, st, max_its, enqueue);
  return finish_solve(op, cb, rc, x->d, diag, /*peer=*/true, history, hist_len, last_step, last_value);
}

}  // namespace bp5
