// Peer-memory transport for the domain-partitioned layout: one process per GPU, every exchange of the CG
// iteration done by kernels that store straight into the neighbour's memory over NVLink / NVSwitch
// (CUDA IPC mappings), with flags instead of host synchronisation.
//
// Replaces, for blocks inside one NVSwitch domain, what the reference does through
// Utilities::MPI::Partitioner + CUDA-aware MPI inside MatrixFree::cell_loop [UPSTREAM]
// (update_ghost_values_start/finish, compress_start/finish with overlap, bp5/step-64.cu:241) and the
// per-iteration cudaMemcpy + MPI_Allreduce of seven doubles (bp5/solver.h:489-494):
//
//   forward   update_ghost_values(d):  the owner's pack kernel writes its upper face / edge / corner values
//             directly into the upper neighbours' ghost segments of d, then raises their "fwd" flags;
//   boundary  cells that touch a ghost layer run as soon as the fwd flags are up (tiles [0, n_boundary_tiles));
//   reverse   compress(add)(h): the ghost segments of h (contributions for the owners) are stored into the
//             lower neighbours' landing zones, "rev" flags raised; the interior cells -- all the others --
//             run while that is in flight; the owner then adds the landing zone onto its upper faces;
//   sums      each rank stores its seven local sums into every rank's mailbox; every rank adds the
//             mailboxes in rank order (bitwise identical everywhere) and runs the scalar recurrences.
// Flags carry a monotonically increasing epoch; a flag doubles as the acknowledgement that frees the
// buffer of the opposite direction (see the ordering argument in DESIGN.md section 6).
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "cg_state.cuh"
#include "common.h"

namespace bp5 {

constexpr int kPeerMaxWorld = 64;

struct PeerLayout {                       // offsets (in doubles) inside the peer buffer
  long long recv_rev;                     // [n_send] landing zone of compress(add)
  long long mailbox;                      // [2][kPeerMaxWorld][8] sums
  long long flags;                        // int32: fwd[8] | rev[8] | sum[2][kPeerMaxWorld]
  long long total;
};
static PeerLayout peer_layout(long long n_send) {
  PeerLayout L;
  L.recv_rev = 0;
  L.mailbox = (n_send + 15) & ~15LL;
  L.flags = L.mailbox + 2LL * kPeerMaxWorld * 8;
  L.total = L.flags + (16 + 2 * kPeerMaxWorld + 1) / 2 + 16;
  return L;
}

struct PeerState {
  int rank = 0, world = 1;
  double *buf = nullptr;                  // own peer buffer
  PeerLayout lay{};
  long long n_send = 0;
  void *mapped[kPeerMaxWorld] = {nullptr};        // peer buffers of the other ranks (IPC mappings), own at [rank]
  void *mapped_d[8] = {nullptr};                  // d vectors of the upper neighbours m = 1..7
  double *fwd_dst[8] = {nullptr};                 // where send group m lands: upper(m)'s ghost segment of d
  int *fwd_flag[8] = {nullptr};                   // upper(m)'s fwd flag m
  double *rev_dst[8] = {nullptr};                 // where ghost group m lands: lower(m)'s recv_rev segment
  int *rev_flag[8] = {nullptr};                   // lower(m)'s rev flag m
  // device words: [0],[1] tickets for "last block" detection; [2] halo epoch = exchanges executed;
  // [3] sum epoch = allreduces executed; [4] error latch (a wait timed out).  The epochs live on the device and only advance when the kernel
  // really runs (not when the CG has converged and every kernel is a no-op), so they stay equal on all
  // ranks even though the hosts may enqueue different numbers of no-op iterations.
  unsigned *ticket = nullptr;
  long long peer_mailbox_off[kPeerMaxWorld] = {0};   // layout of every rank's buffer (depends on its n_send)
  long long peer_flags_off[kPeerMaxWorld] = {0};
  double *scratch = nullptr;              // [16] device: local sums in, global sums out
};

static int *flag_ptr(double *buf, const PeerLayout &L) { return reinterpret_cast<int *>(buf + L.flags); }

__device__ __forceinline__ void st_release_sys(int *p, int v) {
  asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_sys(const int *p) {
  int v;
  asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Wait until *flag has reached `epoch`.  A neighbour that died (or a caller that broke the collective call
// order) must not hang this GPU: after kPeerTimeoutNs the wait gives up, latches *err, and every later wait
// returns at once; the host reports the failure when the solve ends (peer_check).
// default 20 s, BP5_PEER_TIMEOUT_S overrides (read when the transport is connected)
__device__ unsigned long long g_peer_timeout_ns = 20ull * 1000 * 1000 * 1000;
__device__ __forceinline__ void spin_until(const int *flag, int epoch, unsigned *err) {
  const unsigned long long kPeerTimeoutNs = g_peer_timeout_ns;
  if (*reinterpret_cast<volatile unsigned *>(err) != 0) return;
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  unsigned spins = 0;
  while (ld_acquire_sys(flag) - epoch < 0) {
    __nanosleep(64);
    if ((++spins & 1023u) == 0) {
      unsigned long long t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > kPeerTimeoutNs) { atomicExch(err, 1u); return; }
    }
  }
}

struct PeerSendGeom {
  int od[3];
  long long count[8], offset[8];          // send groups (upper neighbours), packed order
  long long gcount[8], goffset[8];        // ghost groups (lower neighbours), offsets relative to n_owned
  long long n_owned;
  double *fwd_dst[8];
  int *fwd_flag[8];
  double *rev_dst[8];
  int *rev_flag[8];
};

__device__ __forceinline__ long long peer_send_index(const PeerSendGeom &g, int m, long long t) {
  int q[3];
  long long rem = t;
  for (int d = 0; d < 3; ++d) {
    if (m & (1 << d)) q[d] = g.od[d] - 1;
    else { q[d] = (int)(rem % g.od[d]); rem /= g.od[d]; }
  }
  return q[0] + (long long)g.od[0] * (q[1] + (long long)g.od[1] * q[2]);
}

// all stores of the grid are globally visible before the flags go up: every block fences and takes a
// ticket; the last one raises the flags
__device__ __forceinline__ bool grid_last_block(unsigned *ticket) {
  __shared__ bool last;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(ticket, 1u);
    last = (t == gridDim.x - 1);
    if (last) {
      *ticket = 0;
      __threadfence_system();     // acquire side: the other blocks' fenced stores are ordered before what follows
    }
  }
  __syncthreads();
  return last;
}

// forward: owned upper-face values of vec -> the upper neighbours' ghost segments
__global__ void peer_forward_kernel(PeerSendGeom g, const double *__restrict__ vec, long long total, unsigned *ticket,
                                    unsigned *epoch_word, const int *skip) {
  if (skip != nullptr && *skip != 0) return;
  __shared__ int epoch;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int m = 1;
    while (m < 7 && i >= g.offset[m] + g.count[m]) ++m;
    const long long t = i - g.offset[m];
    g.fwd_dst[m][t] = vec[peer_send_index(g, m, t)];
  }
  if (grid_last_block(ticket)) {
    if (threadIdx.x == 0) epoch = (int)(++*epoch_word);       // a new exchange begins (always launched, even empty)
    __syncthreads();
    if (threadIdx.x >= 1 && threadIdx.x < 8 && g.count[threadIdx.x] > 0) st_release_sys(g.fwd_flag[threadIdx.x], epoch);
  }
}

// reverse: own ghost segments of vec (contributions for the owners) -> the lower neighbours' landing zones
__global__ void peer_reverse_kernel(PeerSendGeom g, const double *__restrict__ vec, long long total, unsigned *ticket,
                                    const unsigned *epoch_word, const int *skip) {
  if (skip != nullptr && *skip != 0) return;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int m = 1;
    while (m < 7 && i >= g.goffset[m] + g.gcount[m]) ++m;
    const long long t = i - g.goffset[m];
    g.rev_dst[m][t] = vec[g.n_owned + i];
  }
  if (grid_last_block(ticket) && threadIdx.x >= 1 && threadIdx.x < 8 && g.gcount[threadIdx.x] > 0)
    st_release_sys(g.rev_flag[threadIdx.x], (int)*epoch_word);
}

// wait until the lower neighbours' forward data of this epoch has landed (one thread per group)
__global__ void peer_wait_forward_kernel(PeerSendGeom g, const int *flags, const unsigned *epoch_word, unsigned *err,
                                         const int *skip) {
  if (skip != nullptr && *skip != 0) return;
  const int m = threadIdx.x;
  const int epoch = (int)*epoch_word;
  if (m >= 1 && m < 8 && g.gcount[m] > 0) spin_until(flags + m, epoch, err);
}

// wait for the upper neighbours' contributions, then vec[owned upper faces] += landing zone
__global__ void peer_wait_add_kernel(PeerSendGeom g, double *__restrict__ vec, const double *__restrict__ recv,
                                     long long total, const int *flags, const unsigned *epoch_word, unsigned *err,
                                     const int *skip) {
  if (skip != nullptr && *skip != 0) return;
  const int epoch = (int)*epoch_word;
  if (threadIdx.x >= 1 && threadIdx.x < 8 && g.count[threadIdx.x] > 0) spin_until(flags + 8 + threadIdx.x, epoch, err);
  __syncthreads();
  // different groups can hit the same owned DoF (a corner is in the face, edge and corner groups)
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int m = 1;
    while (m < 7 && i >= g.offset[m] + g.count[m]) ++m;
    atomicAdd(&vec[peer_send_index(g, m, i - g.offset[m])], __ldcg(recv + i));
  }
}

struct PeerSumPtrs {
  double *mailbox[kPeerMaxWorld];   // every rank's mailbox base (own included)
  int *sumflag[kPeerMaxWorld];      // every rank's sum-flag base
};

// One block.  Stores `n_vals` (<= 8) local sums into slot [parity][rank] of every rank's mailbox, raises the
// flags, waits for everybody's, and leaves the rank-ordered total in out[0..n_vals).
// cg != nullptr: the seven sums of a merged-CG iteration -- thread 0 goes on with the scalar recurrences
// (solver.h:497-533) right here instead of in a kernel of its own.
__global__ void peer_allreduce_kernel(PeerSumPtrs pp, const double *__restrict__ local, double *__restrict__ out,
                                      int n_vals, int rank, int world, unsigned *epoch_word, unsigned *err,
                                      const int *skip, CgState *cg, double *history) {
  if (skip != nullptr && *skip != 0) return;
  __shared__ int epoch_sh;
  __shared__ double total_sh[8];
  if (threadIdx.x == 0) epoch_sh = (int)(++*epoch_word);
  __syncthreads();
  const int epoch = epoch_sh;
  const int parity = epoch & 1;     // strictly alternating: slot [parity] is free again once everybody's flag of
                                    // epoch - 1 has been seen, which they raise after reading epoch - 2
  const int t = threadIdx.x;
  if (t < world * 8) {
    const int r = t / 8, j = t % 8;
    if (j < n_vals) pp.mailbox[r][(parity * kPeerMaxWorld + rank) * 8 + j] = local[j];
  }
  __threadfence_system();
  __syncthreads();
  if (t < world) st_release_sys(pp.sumflag[t] + parity * kPeerMaxWorld + rank, epoch);
  if (t < world) {
    spin_until(pp.sumflag[rank] + parity * kPeerMaxWorld + t, epoch, err);
  }
  __syncthreads();
  if (t < n_vals) {
    double s = 0.0;
    const double *mb = pp.mailbox[rank] + (long long)parity * kPeerMaxWorld * 8;
    for (int r = 0; r < world; ++r) s += __ldcg(mb + r * 8 + t);     // rank order: identical on every rank
    out[t] = s;
    total_sh[t] = s;
  }
  if (cg != nullptr) {
    __syncthreads();
    if (t == 0) {
      double q[7];
#pragma unroll
      for (int j = 0; j < 7; ++j) q[j] = total_sh[j];
      cg_scalar_step(cg, q, history);
    }
  }
}

static PeerSendGeom make_geom(bp5_operator_t op, const PeerState *ps) {
  PeerSendGeom g{};
  for (int d = 0; d < 3; ++d) g.od[d] = op->od[d];
  int64_t sc[8], so[8], rc[8], ro[8];
  halo_info(op, sc, so, rc, ro);
  for (int m = 0; m < 8; ++m) {
    g.count[m] = sc[m]; g.offset[m] = so[m]; g.gcount[m] = rc[m]; g.goffset[m] = ro[m];
    g.fwd_dst[m] = ps->fwd_dst[m]; g.fwd_flag[m] = ps->fwd_flag[m];
    g.rev_dst[m] = ps->rev_dst[m]; g.rev_flag[m] = ps->rev_flag[m];
  }
  g.n_owned = op->n_owned;
  return g;
}

static unsigned copy_grid(long long total) {
  long long grid = (total + 255) / 256;
  if (grid > 148 * 4) grid = 148 * 4;
  if (grid < 1) grid = 1;
  return (unsigned)grid;
}

// ------------------------------------------------------------------ host entry points (called from abi.cu)
int peer_export(bp5_operator_t op, int rank, int world, bp5_peer_info_t *out) {
  BP5_REQUIRE(world >= 1 && world <= kPeerMaxWorld && rank >= 0 && rank < world, "bad rank / world size");
  bp5_context_t ctx = op->ctx;
  int rc;
  if ((rc = cg_buffers(op, 0, nullptr))) return rc;   // the CG work vectors double as the exchange vectors
  if (!op->peer) {
    PeerState *ps = new PeerState;
    int64_t sc[8], so[8], rcv[8], ro[8];
    halo_info(op, sc, so, rcv, ro);
    ps->n_send = so[7] + sc[7];
    ps->lay = peer_layout(ps->n_send);
    ps->rank = rank; ps->world = world;
    BP5_CUDA(cudaMalloc(&ps->buf, sizeof(double) * ps->lay.total));
    BP5_CUDA(cudaMemset(ps->buf, 0, sizeof(double) * ps->lay.total));
    BP5_CUDA(cudaMalloc(&ps->ticket, sizeof(unsigned) * 8));
    BP5_CUDA(cudaMemset(ps->ticket, 0, sizeof(unsigned) * 8));
    BP5_CUDA(cudaMalloc(&ps->scratch, sizeof(double) * 16));
    BP5_CUDA(cudaMemset(ps->scratch, 0, sizeof(double) * 16));
    BP5_CUDA(cudaDeviceSynchronize());   // the memsets ran on the default stream; everything else uses ctx->stream
    op->peer = ps;
  }
  PeerState *ps = static_cast<PeerState *>(op->peer);
  std::memset(out, 0, sizeof(*out));
  cudaIpcMemHandle_t hb, hd;
  BP5_CUDA(cudaIpcGetMemHandle(&hb, ps->buf));
  BP5_CUDA(cudaIpcGetMemHandle(&hd, op->d->d));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  std::memcpy(out->buf_handle, &hb, 64);
  std::memcpy(out->dvec_handle, &hd, 64);
  out->n_owned = op->n_owned; out->n_ghost = op->n_ghost;
  int64_t sc[8], so[8], rcv[8], ro[8];
  halo_info(op, sc, so, rcv, ro);
  for (int m = 0; m < 8; ++m) { out->ghost_offset[m] = ro[m]; out->send_offset[m] = so[m]; }
  out->n_send = ps->n_send;
  out->rank = rank;
  out->device = ctx->device;
  return BP5_OK;
}

int peer_connect(bp5_operator_t op, const bp5_peer_info_t *all, const int *upper_rank, const int *lower_rank) {
  BP5_REQUIRE(op->peer, "bp5_peer_export has not been called");
  PeerState *ps = static_cast<PeerState *>(op->peer);
  for (int r = 0; r < ps->world; ++r) {
    const PeerLayout L = peer_layout(all[r].n_send);
    ps->peer_mailbox_off[r] = L.mailbox;
    ps->peer_flags_off[r] = L.flags;
    if (r == ps->rank) { ps->mapped[r] = ps->buf; continue; }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, all[r].buf_handle, 64);
    BP5_CUDA(cudaIpcOpenMemHandle(&ps->mapped[r], h, cudaIpcMemLazyEnablePeerAccess));
  }
  for (int m = 1; m < 8; ++m) {
    const int up = upper_rank[m], lo = lower_rank[m];
    if (up >= 0) {
      BP5_REQUIRE(up < ps->world && up != ps->rank, "bad upper neighbour");
      cudaIpcMemHandle_t h;
      std::memcpy(&h, all[up].dvec_handle, 64);
      // the same neighbour can appear for several m only in degenerate grids; open once per m is fine for
      // distinct ranks, reuse the mapping otherwise
      void *base = nullptr;
      for (int k = 1; k < m; ++k)
        if (upper_rank[k] == up) base = ps->mapped_d[k];
      if (!base) BP5_CUDA(cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess));
      ps->mapped_d[m] = base;
      ps->fwd_dst[m] = static_cast<double *>(base) + all[up].n_owned + all[up].ghost_offset[m];
      ps->fwd_flag[m] = flag_ptr(static_cast<double *>(ps->mapped[up]), peer_layout(all[up].n_send)) + m;
    }
    if (lo >= 0) {
      BP5_REQUIRE(lo < ps->world && lo != ps->rank, "bad lower neighbour");
      const PeerLayout L = peer_layout(all[lo].n_send);
      ps->rev_dst[m] = static_cast<double *>(ps->mapped[lo]) + L.recv_rev + all[lo].send_offset[m];
      ps->rev_flag[m] = flag_ptr(static_cast<double *>(ps->mapped[lo]), L) + 8 + m;
    }
  }
  if (const char *tv = getenv("BP5_PEER_TIMEOUT_S")) {
    const unsigned long long ns = (unsigned long long)(std::max(1.0, atof(tv)) * 1e9);
    BP5_CUDA(cudaMemcpyToSymbol(g_peer_timeout_ns, &ns, sizeof(ns)));
  }
  op->peer_connected = true;
  return BP5_OK;
}

void peer_destroy(bp5_operator_t op) {
  if (!op->peer) return;
  PeerState *ps = static_cast<PeerState *>(op->peer);
  for (int r = 0; r < ps->world; ++r)
    if (r != ps->rank && ps->mapped[r]) cudaIpcCloseMemHandle(ps->mapped[r]);
  for (int m = 1; m < 8; ++m) {
    bool dup = false;
    for (int k = 1; k < m; ++k) dup |= ps->mapped_d[k] == ps->mapped_d[m];
    if (ps->mapped_d[m] && !dup) cudaIpcCloseMemHandle(ps->mapped_d[m]);
  }
  cudaFree(ps->buf);
  cudaFree(ps->ticket);
  cudaFree(ps->scratch);
  delete ps;
  op->peer = nullptr;
}

// update_ghost_values(d), sender half + receiver wait
int peer_wait_forward(bp5_operator_t op) {
  PeerState *ps = static_cast<PeerState *>(op->peer);
  if (op->n_ghost == 0) return BP5_OK;
  const PeerSendGeom g = make_geom(op, ps);
  peer_wait_forward_kernel<<<1, 32, 0, op->ctx->stream>>>(g, flag_ptr(ps->buf, ps->lay), ps->ticket + 2, ps->ticket + 4,
                                                         op->skip_flag);
  BP5_CHECK_LAUNCH();
  op->ctx->launches++;
  return BP5_OK;
}

int peer_forward(bp5_operator_t op, const double *vec_owned_of_d, bool wait) {
  PeerState *ps = static_cast<PeerState *>(op->peer);
  const PeerSendGeom g = make_geom(op, ps);
  cudaStream_t s = op->ctx->stream;
  // always launched: it also opens the exchange (advances the halo epoch)
  peer_forward_kernel<<<copy_grid(ps->n_send), 256, 0, s>>>(g, vec_owned_of_d, ps->n_send, ps->ticket, ps->ticket + 2,
                                                           op->skip_flag);
  BP5_CHECK_LAUNCH();
  op->ctx->launches++;
  return wait ? peer_wait_forward(op) : BP5_OK;
}

// compress(add)(h), sender half
int peer_reverse(bp5_operator_t op, const double *vec) {
  PeerState *ps = static_cast<PeerState *>(op->peer);
  if (op->n_ghost == 0) return BP5_OK;
  const PeerSendGeom g = make_geom(op, ps);
  peer_reverse_kernel<<<copy_grid(op->n_ghost), 256, 0, op->ctx->stream>>>(g, vec, op->n_ghost, ps->ticket + 1,
                                                                          ps->ticket + 2, op->skip_flag);
  BP5_CHECK_LAUNCH();
  op->ctx->launches++;
  return BP5_OK;
}

// compress(add)(h), owner half: wait for the contributions, add them
int peer_wait_add(bp5_operator_t op, double *vec) {
  PeerState *ps = static_cast<PeerState *>(op->peer);
  if (ps->n_send == 0) return BP5_OK;
  const PeerSendGeom g = make_geom(op, ps);
  peer_wait_add_kernel<<<copy_grid(ps->n_send), 256, 0, op->ctx->stream>>>(
      g, vec, ps->buf + ps->lay.recv_rev, ps->n_send, flag_ptr(ps->buf, ps->lay), ps->ticket + 2, ps->ticket + 4,
      op->skip_flag);
  BP5_CHECK_LAUNCH();
  op->ctx->launches++;
  return BP5_OK;
}

// sum of n_vals doubles over all ranks, device to device
int peer_allreduce(bp5_operator_t op, const double *local_dev, double *out_dev, int n_vals, bool honour_skip,
                   void *cg_state, double *history) {
  PeerState *ps = static_cast<PeerState *>(op->peer);
  BP5_REQUIRE(n_vals >= 1 && n_vals <= 8, "1..8 values");
  PeerSumPtrs pp{};
  for (int r = 0; r < ps->world; ++r) {
    double *base = static_cast<double *>(ps->mapped[r]);
    // every rank allocates the same layout family; the mailbox offset depends on that rank's n_send
    pp.mailbox[r] = base + ps->peer_mailbox_off[r];
    pp.sumflag[r] = reinterpret_cast<int *>(base + ps->peer_flags_off[r]) + 16;
  }
  const int threads = ((ps->world * 8 + 31) / 32) * 32;
  peer_allreduce_kernel<<<1, threads, 0, op->ctx->stream>>>(pp, local_dev, out_dev, n_vals, ps->rank, ps->world,
                                                           ps->ticket + 3, ps->ticket + 4,
                                                           honour_skip ? op->skip_flag : nullptr,
                                                           static_cast<CgState *>(cg_state), history);
  BP5_CHECK_LAUNCH();
  op->ctx->launches++;
  return BP5_OK;
}

}  // namespace bp5

namespace bp5 {
double *peer_scratch(bp5_operator_t op) { return static_cast<PeerState *>(op->peer)->scratch; }

// after a collective call has been synchronised: did any wait give up?
int peer_check(bp5_operator_t op) {
  PeerState *ps = static_cast<PeerState *>(op->peer);
  unsigned err = 0;
  BP5_CUDA(cudaMemcpyAsync(&err, ps->ticket + 4, sizeof(unsigned), cudaMemcpyDeviceToHost, op->ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(op->ctx->stream));
  if (err != 0) {
    // reported once: re-arm the latch so that a later, correctly ordered collective call can succeed (the flags and
    // epochs of the call that timed out are undefined, the caller should re-create the operator to be safe)
    BP5_CUDA(cudaMemsetAsync(ps->ticket + 4, 0, sizeof(unsigned), op->ctx->stream));
    set_error("peer exchange timed out: a neighbouring rank did not reach the same collective call within "
              "BP5_PEER_TIMEOUT_S (default 20 s); ranks must enter collective calls together (barrier after connect)");
    return BP5_ERR_CUDA;
  }
  return BP5_OK;
}

// sum over all ranks of n host values (norms, parity checks): host -> device -> peers -> host
int peer_allreduce_host(bp5_operator_t op, double *vals, int n) {
  BP5_REQUIRE(op->peer && op->peer_connected, "peer transport not connected");
  BP5_REQUIRE(n >= 1 && n <= 8, "1..8 values");
  PeerState *ps = static_cast<PeerState *>(op->peer);
  cudaStream_t s = op->ctx->stream;
  BP5_CUDA(cudaMemcpyAsync(ps->scratch, vals, sizeof(double) * n, cudaMemcpyHostToDevice, s));
  int rc;
  if ((rc = peer_allreduce(op, ps->scratch, ps->scratch + 8, n, false, nullptr, nullptr))) return rc;
  BP5_CUDA(cudaMemcpyAsync(vals, ps->scratch + 8, sizeof(double) * n, cudaMemcpyDeviceToHost, s));
  BP5_CUDA(cudaStreamSynchronize(s));
  return peer_check(op);
}

int peer_world_size(bp5_operator_t op) {
  if (!op->peer || !op->peer_connected) return 1;
  return static_cast<PeerState *>(op->peer)->world;
}

// Stand-alone ghost operations on any vector of the operator's layout.  Each one is a complete exchange round
// (forward, consume, reverse, add) so that the flag / epoch protocol of the CG loop -- where the flag of one
// direction acknowledges the buffer of the other -- stays intact whatever sequence of calls the host makes.
// update_ghost_values: the forward half carries the data (it lands in the neighbour's ghost segment of ITS d
// vector, from where that rank copies it into its vector); the reverse half carries zeros.
int peer_update_ghost_values(bp5_operator_t op, bp5_vector_t vec) {
  BP5_REQUIRE(op->peer && op->peer_connected, "peer transport not connected");
  cudaStream_t s = op->ctx->stream;
  int rc;
  if ((rc = peer_forward(op, vec->d))) return rc;
  if (op->n_ghost > 0 && vec->d != op->d->d)
    BP5_CUDA(cudaMemcpyAsync(vec->d + op->n_owned, op->d->d + op->n_owned, sizeof(double) * op->n_ghost,
                             cudaMemcpyDeviceToDevice, s));
  if (op->n_ghost > 0) BP5_CUDA(cudaMemsetAsync(op->h->d + op->n_owned, 0, sizeof(double) * op->n_ghost, s));
  if ((rc = peer_reverse(op, op->h->d))) return rc;
  return peer_wait_add(op, op->h->d);              // adds zeros onto the scratch vector's faces
}

// compress(add): the forward half carries nothing of interest, the reverse half the ghost contributions
int peer_compress_add(bp5_operator_t op, bp5_vector_t vec) {
  BP5_REQUIRE(op->peer && op->peer_connected, "peer transport not connected");
  int rc;
  if ((rc = peer_forward(op, op->d->d))) return rc;
  if ((rc = peer_reverse(op, vec->d))) return rc;
  if ((rc = peer_wait_add(op, vec->d))) return rc;
  if (op->n_ghost > 0)
    BP5_CUDA(cudaMemsetAsync(vec->d + op->n_owned, 0, sizeof(double) * op->n_ghost, op->ctx->stream));
  return BP5_OK;
}

// PoissonOperator::vmult over the partition through the peer transport (bp5/step-64.cu:263-276 with the
// exchanges of MatrixFree::cell_loop): dst = A src on the owned range.  The exchange vectors are the
// operator's own d / h (their ghost segments are what the neighbours are mapped to).
int peer_vmult(bp5_operator_t op, bp5_vector_t dst, bp5_vector_t src) {
  BP5_REQUIRE(op->peer && op->peer_connected, "peer transport not connected");
  cudaStream_t s = op->ctx->stream;
  const size_t owned_bytes = sizeof(double) * op->n_owned;
  int rc;
  BP5_CUDA(cudaMemcpyAsync(op->d->d, src->d, owned_bytes, cudaMemcpyDeviceToDevice, s));
  BP5_CUDA(cudaMemsetAsync(op->h->d, 0, sizeof(double) * (op->n_owned + op->n_ghost), s));
  if ((rc = peer_forward(op, op->d->d))) return rc;
  if ((rc = apply_cell_loop(op, op->h->d, op->d->d, false, nullptr, 1))) return rc;
  if ((rc = peer_reverse(op, op->h->d))) return rc;
  if ((rc = apply_cell_loop(op, op->h->d, op->d->d, false, nullptr, 2))) return rc;
  if ((rc = peer_wait_add(op, op->h->d))) return rc;
  BP5_CUDA(cudaMemcpyAsync(dst->d, op->h->d, owned_bytes, cudaMemcpyDeviceToDevice, s));
  return apply_copy_constrained(op, dst->d, src->d);
}
}  // namespace bp5
