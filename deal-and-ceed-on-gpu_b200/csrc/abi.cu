// extern "C" entry points declared in include/bp5_b200.h.
#include <cstring>
#include <new>

#include "common.h"

namespace bp5 {
static thread_local char g_error[1024] = "";
void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}
const char *get_error() { return g_error; }
}  // namespace bp5

using namespace bp5;

#define BP5_ABI_GUARD_BEGIN try {
#define BP5_ABI_GUARD_END                                     \
  }                                                           \
  catch (const std::bad_alloc &) {                            \
    set_error("out of host memory");                          \
    return BP5_ERR_INVALID;                                   \
  }                                                           \
  catch (...) {                                               \
    set_error("unexpected C++ exception at the ABI boundary"); \
    return BP5_ERR_INVALID;                                   \
  }

// Host-buffer solves: b and the owned range of x (or zeros when x0_is_zero) go to the operator's staging vectors, whose
// ghost entries are zero; `solve(x, b)` runs on them, and x comes back unless the solve failed outright.
template <typename Solve>
static int solve_host(bp5_operator_t op, double *x_host, const double *b_host, int x0_is_zero, Solve solve) {
  bp5_context_t ctx = op->ctx;
  const int64_t n = op->n_owned;
  int rc;
  if (!op->xh) {
    if ((rc = bp5_vector_create(ctx, op->n_owned, op->n_ghost, &op->xh))) return rc;
    if ((rc = bp5_vector_create(ctx, op->n_owned, op->n_ghost, &op->bh))) return rc;
  }
  BP5_CUDA(cudaMemcpyAsync(op->bh->d, b_host, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
  if (x0_is_zero) {
    BP5_CUDA(cudaMemsetAsync(op->xh->d, 0, sizeof(double) * (n + op->n_ghost), ctx->stream));
  } else {
    BP5_CUDA(cudaMemcpyAsync(op->xh->d, x_host, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
    if (op->n_ghost) BP5_CUDA(cudaMemsetAsync(op->xh->d + n, 0, sizeof(double) * op->n_ghost, ctx->stream));
  }
  rc = solve(op->xh, op->bh);
  if (rc != BP5_OK && rc != BP5_ERR_NO_CONVERGENCE) return rc;
  BP5_CUDA(cudaMemcpyAsync(x_host, op->xh->d, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  return rc;
}

extern "C" {

const char *bp5_last_error(void) { return get_error(); }
const char *bp5_version(void) { return "bp5_b200 0.1 (sm_100a)"; }

// ------------------------------------------------------------------ context
int bp5_context_create(int device, bp5_context_t *out) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(out != nullptr, "null output pointer");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    set_error("no CUDA device available (%s); this library has no CPU fallback",
              e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return BP5_ERR_CUDA;
  }
  BP5_REQUIRE(device >= 0 && device < count, "device index out of range");
  BP5_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  BP5_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    return BP5_ERR_UNSUPPORTED;
  }
  bp5_context_t ctx = new bp5_context_s;
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  BP5_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  BP5_CUDA(cudaMalloc(&ctx->scratch, sizeof(double) * 1024));
  BP5_CUDA(cudaMallocHost(&ctx->scratch_host, sizeof(double) * 64));
  *out = ctx;
  return BP5_OK;
  BP5_ABI_GUARD_END
}

int bp5_context_destroy(bp5_context_t ctx) {
  if (!ctx) return BP5_OK;
  cudaSetDevice(ctx->device);
  if (ctx->stream) { cudaStreamSynchronize(ctx->stream); cudaStreamDestroy(ctx->stream); }
  cudaFree(ctx->scratch);
  cudaFreeHost(ctx->scratch_host);
  delete ctx;
  return BP5_OK;
}

int bp5_context_synchronize(bp5_context_t ctx) {
  BP5_REQUIRE(ctx, "null context");
  BP5_CUDA(cudaStreamSynchronize(ctx->stream));
  return BP5_OK;
}
void *bp5_context_stream(bp5_context_t ctx) { return ctx ? (void *)ctx->stream : nullptr; }
int64_t bp5_context_launch_count(bp5_context_t ctx) { return ctx ? ctx->launches : 0; }

// ----------------------------------------------------------------- operator
int bp5_operator_create(bp5_context_t ctx, const bp5_problem_t *pr, bp5_operator_t *out) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(ctx && pr && out, "null argument");
  BP5_REQUIRE(pr->degree >= 1 && pr->degree <= kMaxDegree, "degree must be in 1..8");
  BP5_REQUIRE(pr->quadrature == BP5_QUAD_GAUSS || pr->quadrature == BP5_QUAD_GLL, "unknown quadrature");
  BP5_REQUIRE(pr->operator_kind == BP5_OP_POISSON || pr->operator_kind == BP5_OP_HELMHOLTZ, "unknown operator");
  BP5_REQUIRE(pr->geometry_mode == BP5_GEOM_STORED || pr->geometry_mode == BP5_GEOM_ON_THE_FLY, "unknown geometry mode");
  BP5_REQUIRE(pr->deformation == 0 || pr->deformation == 1, "unknown deformation");
  BP5_REQUIRE(pr->cell_order == BP5_CELL_ORDER_DEFAULT || pr->cell_order == BP5_CELL_ORDER_COLORED, "unknown cell order");
  BP5_REQUIRE(pr->reserved[0] == 0, "reserved fields of bp5_problem_t must be zero");
  bool refined = false, refine_set = false;
  for (int d = 0; d < 3; ++d) refine_set |= pr->refine_lo[d] != 0 || pr->refine_hi[d] != 0;
  if (refine_set) {
    for (int d = 0; d < 3; ++d)
      BP5_REQUIRE(pr->refine_lo[d] >= 0 && pr->refine_lo[d] < pr->refine_hi[d] && pr->refine_hi[d] <= pr->cells[d],
                  "refine box must satisfy 0 <= refine_lo < refine_hi <= cells in every direction");
    refined = true;
    if (pr->geometry_mode != BP5_GEOM_STORED || pr->cell_order != BP5_CELL_ORDER_DEFAULT ||
        pr->part_grid[0] * pr->part_grid[1] * pr->part_grid[2] != 1) {
      set_error("locally refined meshes are implemented for one block with stored geometry and the default cell order");
      return BP5_ERR_UNSUPPORTED;
    }
  }
  if (pr->cell_order == BP5_CELL_ORDER_COLORED &&
      (pr->geometry_mode != BP5_GEOM_STORED || pr->part_grid[0] * pr->part_grid[1] * pr->part_grid[2] != 1)) {
    set_error("the coloured cell order is implemented for one block with stored geometry");
    return BP5_ERR_UNSUPPORTED;
  }
  for (int d = 0; d < 3; ++d) {
    BP5_REQUIRE(pr->cells[d] >= 1, "cells must be >= 1");
    BP5_REQUIRE(pr->upper[d] > pr->lower[d], "upper must exceed lower");
    BP5_REQUIRE(pr->part_grid[d] >= 1 && pr->part_coord[d] >= 0 && pr->part_coord[d] < pr->part_grid[d],
                "bad partition");
    BP5_REQUIRE(pr->part_grid[d] <= pr->cells[d], "more blocks than cells in a direction");
  }
  BP5_CUDA(cudaSetDevice(ctx->device));
  bp5_operator_t op = new bp5_operator_s;
  op->ctx = ctx;
  op->prob = *pr;
  op->p = pr->degree;
  op->n = pr->degree + 1;
  make_tables(op->p, pr->quadrature, op->tab);
  op->metric_planes = pr->operator_kind == BP5_OP_HELMHOLTZ ? 7 : 6;
  int64_t owned = 1, ncell = 1, nglob = 1;
  for (int d = 0; d < 3; ++d) {
    const int64_t G = pr->cells[d], P = pr->part_grid[d], c = pr->part_coord[d];
    op->c0[d] = (int)(G * c / P);
    op->lc[d] = (int)(G * (c + 1) / P) - op->c0[d];
    op->ld[d] = op->lc[d] * op->p + 1;
    op->has_lo[d] = c > 0;
    op->has_hi[d] = c < P - 1;
    op->od[d] = op->ld[d] - op->has_lo[d];
    owned *= op->od[d];
    ncell *= op->lc[d];
    nglob *= G * op->p + 1;
  }
  op->n_owned = owned;
  op->n_cells = ncell;
  op->n_global = nglob;
  int64_t goff = 0;
  for (int m = 1; m < 8; ++m) {
    bool exists = true;
    int64_t sz = 1;
    for (int d = 0; d < 3; ++d) {
      if (m & (1 << d)) { if (!op->has_lo[d]) exists = false; }
      else sz *= op->od[d];
    }
    op->ghost_offset[m] = goff;
    op->ghost_size[m] = exists ? sz : 0;
    goff += op->ghost_size[m];
  }
  op->n_ghost = goff;
  if (op->n_owned + op->n_ghost >= (int64_t)2147483647) {
    delete op;
    set_error("block has %lld local DoFs; local indices are 32-bit (types::global_dof_index default)",
              (long long)(owned + goff));
    return BP5_ERR_UNSUPPORTED;
  }
  int rc;
  if (refined) {
    // hanging nodes: numbering and the generic functor path's arrays only (the tuned kernel handles conforming meshes)
    rc = operator_setup_hanging(op);
  } else {
    rc = apply_choose(op);
    if (rc == BP5_OK) rc = operator_setup_device(op);
  }
  if (rc != BP5_OK) { bp5_operator_destroy(op); return rc; }
  *out = op;
  return BP5_OK;
  BP5_ABI_GUARD_END
}

int bp5_operator_destroy(bp5_operator_t op) {
  if (!op) return BP5_OK;
  cudaSetDevice(op->ctx->device);
  cudaStreamSynchronize(op->ctx->stream);
  peer_destroy(op);
  cudaFree(op->cell_base);
  cudaFree(op->cell_mask);
  cudaFree(op->hanging_cells);
  cudaFree(op->hanging_interp_dev);
  cudaFree(op->l2g_irr);
  cudaFree(op->mf_l2g); cudaFree(op->mf_constraint_mask); cudaFree(op->mf_inv_jacobian);
  cudaFree(op->mf_jxw); cudaFree(op->mf_q_points);
  for (int c = 0; c < 8; ++c) {
    cudaFree(op->mfc_l2g[c]); cudaFree(op->mfc_constraint_mask[c]); cudaFree(op->mfc_inv_jacobian[c]);
    cudaFree(op->mfc_jxw[c]); cudaFree(op->mfc_q_points[c]);
  }
  cudaFree(op->metric);
  cudaFree(op->coords);
  cudaFree(op->constrained);
  cudaFree(op->cg_scalars);
  for (cudaEvent_t e : op->prof_events) cudaEventDestroy(e);
  bp5_vector_destroy(op->g);
  bp5_vector_destroy(op->d);
  bp5_vector_destroy(op->h);
  bp5_vector_destroy(op->xh);
  bp5_vector_destroy(op->bh);
  delete op;
  return BP5_OK;
}

int bp5_operator_sizes(bp5_operator_t op, int64_t *n_owned, int64_t *n_ghost, int64_t *n_global, int64_t *n_cells) {
  BP5_REQUIRE(op, "null operator");
  if (n_owned) *n_owned = op->n_owned;
  if (n_ghost) *n_ghost = op->n_ghost;
  if (n_global) *n_global = op->n_global;
  if (n_cells) *n_cells = op->n_cells;
  return BP5_OK;
}

int bp5_operator_initialize_dof_vector(bp5_operator_t op, bp5_vector_t *vec) {
  BP5_REQUIRE(op && vec, "null argument");
  const int rc = bp5_vector_create(op->ctx, op->n_owned, op->n_ghost, vec);
  if (rc == BP5_OK) (*vec)->owner = op;
  return rc;
}

int bp5_operator_set_zero_out(bp5_operator_t op, int z) {
  BP5_REQUIRE(op, "null operator");
  op->do_zero_out = z != 0;
  return BP5_OK;
}

// entry points that exist for conforming meshes only
#define BP5_CONFORMING_ONLY(op)                                                                                        \
  do {                                                                                                                 \
    if ((op)->hanging) {                                                                                               \
      set_error("%s is not implemented for locally refined meshes (available there: vmult, cell_loop, the CG "      \
                "solves, assemble_rhs, l2_norm, the diagonal, vectors, bp5_operator_matrix_free_data)"       ,         \
                __func__);                                                                                             \
      return BP5_ERR_UNSUPPORTED;                                                                                      \
    }                                                                                                                  \
  } while (0)

static int check_vec(bp5_operator_t op, bp5_vector_t v) {
  BP5_REQUIRE(v != nullptr, "null vector");
  BP5_REQUIRE(v->n_owned == op->n_owned && v->n_ghost == op->n_ghost, "vector layout does not match the operator");
  return BP5_OK;
}

int bp5_operator_cell_loop(bp5_operator_t op, bp5_vector_t dst, bp5_vector_t src) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op, "null operator");
  int rc;
  if ((rc = check_vec(op, dst)) || (rc = check_vec(op, src))) return rc;
  BP5_REQUIRE(dst != src, "dst and src must differ");
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return apply_cell_loop(op, dst->d, src->d, /*overwrite_interior=*/false);   // dst += A src
  BP5_ABI_GUARD_END
}

int bp5_operator_copy_constrained_values(bp5_operator_t op, bp5_vector_t dst, bp5_vector_t src) {
  BP5_REQUIRE(op, "null operator");
  int rc;
  if ((rc = check_vec(op, dst)) || (rc = check_vec(op, src))) return rc;
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return apply_copy_constrained(op, dst->d, src->d);
}

int bp5_operator_vmult(bp5_operator_t op, bp5_vector_t dst, bp5_vector_t src) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op, "null operator");
  int rc;
  if ((rc = check_vec(op, dst)) || (rc = check_vec(op, src))) return rc;
  BP5_REQUIRE(dst != src, "dst and src must differ");
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  // bp5/step-64.cu:270-275.  With ghosts, the halo exchange is driven by the
  // host that owns the communicator (see INTEGRATION.md); this entry point
  // does the local part: src ghosts must be up to date, dst ghosts receive the
  // contributions for the neighbouring owners.
  // "dst = 0" only has to reach the DoFs shared between cells: cell-interior
  // DoFs receive exactly one contribution and are stored by the kernel.
  if (op->do_zero_out && (rc = apply_zero_skeleton(op, dst->d))) return rc;
  if ((rc = apply_cell_loop(op, dst->d, src->d, /*overwrite_interior=*/op->do_zero_out))) return rc;
  return apply_copy_constrained(op, dst->d, src->d);
  BP5_ABI_GUARD_END
}

int bp5_operator_vmult_ptr(bp5_operator_t op, double *dst, const double *src, int zero_dst) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && dst && src && dst != src, "bad argument");
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  int rc;
  if (zero_dst && (rc = apply_zero_skeleton(op, dst))) return rc;
  if ((rc = apply_cell_loop(op, dst, src, zero_dst != 0))) return rc;
  return apply_copy_constrained(op, dst, src);
  BP5_ABI_GUARD_END
}

int bp5_operator_assemble_rhs(bp5_operator_t op, bp5_vector_t b) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op, "null operator");
  int rc;
  if ((rc = check_vec(op, b))) return rc;
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return operator_assemble_rhs(op, b->d);
  BP5_ABI_GUARD_END
}

int bp5_operator_export_coefficients(bp5_operator_t op, double *host_out) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && host_out, "null argument");
  BP5_CONFORMING_ONLY(op);
  if (!op->metric) { set_error("this operator computes its geometry on the fly: no stored coefficient"); return BP5_ERR_UNSUPPORTED; }
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  BP5_CUDA(cudaStreamSynchronize(op->ctx->stream));
  return operator_export_coefficients(op, host_out);
  BP5_ABI_GUARD_END
}

int bp5_operator_export_dof_coordinates(bp5_operator_t op, double *host_out) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && host_out, "null argument");
  if (op->hanging) { std::copy(op->hanging_coords.begin(), op->hanging_coords.end(), host_out); return BP5_OK; }
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return operator_export_coords(op, host_out);
  BP5_ABI_GUARD_END
}

int bp5_operator_export_global_indices(bp5_operator_t op, int64_t *host_out) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && host_out, "null argument");
  if (op->hanging) { for (int64_t i = 0; i < op->n_owned; ++i) host_out[i] = i; return BP5_OK; }
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return operator_export_global_indices(op, host_out);
  BP5_ABI_GUARD_END
}

int bp5_operator_l2_norm_sqr(bp5_operator_t op, bp5_vector_t u, double *out) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && out, "null argument");
  int rc;
  if ((rc = check_vec(op, u))) return rc;
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return operator_l2_norm_sqr(op, u->d, out);
  BP5_ABI_GUARD_END
}

int bp5_operator_compute_diagonal(bp5_operator_t op, bp5_vector_t diag, int invert) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op, "null operator");
  int rc;
  if ((rc = check_vec(op, diag))) return rc;
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return operator_diagonal(op, diag->d, invert != 0);
  BP5_ABI_GUARD_END
}

int bp5_operator_algorithmic_bytes(bp5_operator_t op, double *per_vmult, double *per_cg_it) {
  BP5_REQUIRE(op, "null operator");
  // SURVEY.md 8(d): per DoF 8 (read src) + 8 (write dst) + 8*planes per q-point;
  // CG: read {x,r,p,h,diag} + write {x,r,p,h} = 72, plus the metric.
  const double n3 = (double)op->n * op->n * op->n;
  // stored metric: 8 bytes per plane per quadrature point; on the fly: three coordinates per local DoF
  const double metric = op->metric_path == 3 ? 0.0        // affine mesh, geometry on the fly: three constants
                        : op->prob.geometry_mode == BP5_GEOM_ON_THE_FLY
                            ? 24.0 * (double)(op->n_owned + op->n_ghost)
                            : 8.0 * op->metric_planes * n3 * (double)op->n_cells;
  if (per_vmult) *per_vmult = 16.0 * (double)op->n_owned + metric;
  if (per_cg_it) *per_cg_it = 72.0 * (double)op->n_owned + metric;
  return BP5_OK;
}

int bp5_operator_profile(bp5_operator_t op, int enable) {
  BP5_REQUIRE(op, "null operator");
  op->profile = enable != 0;
  op->prof_used = 0;
  return BP5_OK;
}

int bp5_operator_profile_result(bp5_operator_t op, int64_t *launches, double *total_ms) {
  BP5_REQUIRE(op && launches && total_ms, "null argument");
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  BP5_CUDA(cudaStreamSynchronize(op->ctx->stream));
  double ms = 0.0;
  for (size_t i = 0; i + 1 < op->prof_used; i += 2) {
    float t = 0.f;
    BP5_CUDA(cudaEventElapsedTime(&t, op->prof_events[i], op->prof_events[i + 1]));
    ms += t;
  }
  *launches = (int64_t)(op->prof_used / 2);
  *total_ms = ms;
  op->prof_used = 0;
  return BP5_OK;
}

const char *bp5_operator_kernel_name(bp5_operator_t op) { return op ? op->kernel_name.c_str() : ""; }

// ------------------------------------------------------------------- vector
int bp5_vector_create(bp5_context_t ctx, int64_t n_owned, int64_t n_ghost, bp5_vector_t *out) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(ctx && out, "null argument");
  BP5_REQUIRE(n_owned >= 0 && n_ghost >= 0, "negative size");
  BP5_CUDA(cudaSetDevice(ctx->device));
  bp5_vector_t v = new bp5_vector_s;
  v->ctx = ctx; v->n_owned = n_owned; v->n_ghost = n_ghost;
  const size_t bytes = sizeof(double) * (size_t)std::max<int64_t>(n_owned + n_ghost, 1);
  cudaError_t e = cudaMalloc(&v->d, bytes);
  if (e != cudaSuccess) {
    delete v;
    set_error("cudaMalloc of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    return BP5_ERR_CUDA;
  }
  // reinit() zero-initialises (solver.h:369-371)
  BP5_CUDA(cudaMemsetAsync(v->d, 0, bytes, ctx->stream));
  *out = v;
  return BP5_OK;
  BP5_ABI_GUARD_END
}

int bp5_vector_create_like(bp5_vector_t other, bp5_vector_t *out) {
  BP5_REQUIRE(other, "null vector");
  const int rc = bp5_vector_create(other->ctx, other->n_owned, other->n_ghost, out);
  if (rc == BP5_OK) (*out)->owner = other->owner;
  return rc;
}

bp5_operator_t bp5_vector_owner(bp5_vector_t v) { return v ? v->owner : nullptr; }

int bp5_vector_destroy(bp5_vector_t v) {
  if (!v) return BP5_OK;
  cudaSetDevice(v->ctx->device);
  cudaStreamSynchronize(v->ctx->stream);
  cudaFree(v->d);
  delete v;
  return BP5_OK;
}

int bp5_vector_local_size(bp5_vector_t v, int64_t *n_owned, int64_t *n_ghost) {
  BP5_REQUIRE(v, "null vector");
  if (n_owned) *n_owned = v->n_owned;
  if (n_ghost) *n_ghost = v->n_ghost;
  return BP5_OK;
}

double *bp5_vector_get_values(bp5_vector_t v) { return v ? v->d : nullptr; }

int bp5_vector_set(bp5_vector_t v, double value) {
  BP5_REQUIRE(v, "null vector");
  BP5_CUDA(cudaSetDevice(v->ctx->device));
  return vec_fill(v->ctx, v->d, v->n_owned + v->n_ghost, value);
}

int bp5_vector_import_host(bp5_vector_t v, const double *host, int64_t n) {
  BP5_REQUIRE(v && host, "null argument");
  BP5_REQUIRE(n >= 0 && n <= v->n_owned + v->n_ghost, "bad length");
  BP5_CUDA(cudaSetDevice(v->ctx->device));
  BP5_CUDA(cudaMemcpyAsync(v->d, host, sizeof(double) * n, cudaMemcpyHostToDevice, v->ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(v->ctx->stream));
  return BP5_OK;
}

int bp5_vector_export_host(bp5_vector_t v, double *host, int64_t n) {
  BP5_REQUIRE(v && host, "null argument");
  BP5_REQUIRE(n >= 0 && n <= v->n_owned + v->n_ghost, "bad length");
  BP5_CUDA(cudaSetDevice(v->ctx->device));
  BP5_CUDA(cudaMemcpyAsync(host, v->d, sizeof(double) * n, cudaMemcpyDeviceToHost, v->ctx->stream));
  BP5_CUDA(cudaStreamSynchronize(v->ctx->stream));
  return BP5_OK;
}

static int same_layout(bp5_vector_t a, bp5_vector_t b) {
  BP5_REQUIRE(a && b, "null vector");
  BP5_REQUIRE(a->n_owned == b->n_owned && a->n_ghost == b->n_ghost, "vector layouts differ");
  return BP5_OK;
}

int bp5_vector_copy(bp5_vector_t dst, bp5_vector_t src) {
  int rc;
  if ((rc = same_layout(dst, src))) return rc;
  BP5_CUDA(cudaSetDevice(dst->ctx->device));
  BP5_CUDA(cudaMemcpyAsync(dst->d, src->d, sizeof(double) * (src->n_owned + src->n_ghost), cudaMemcpyDeviceToDevice,
                           dst->ctx->stream));
  return BP5_OK;
}

int bp5_vector_add(bp5_vector_t y, double a, bp5_vector_t x) {
  int rc;
  if ((rc = same_layout(y, x))) return rc;
  BP5_CUDA(cudaSetDevice(y->ctx->device));
  return vec_axpy(y->ctx, y->d, 1.0, a, x->d, y->n_owned, 0);
}
int bp5_vector_equ(bp5_vector_t y, double a, bp5_vector_t x) {
  int rc;
  if ((rc = same_layout(y, x))) return rc;
  BP5_CUDA(cudaSetDevice(y->ctx->device));
  return vec_axpy(y->ctx, y->d, 0.0, a, x->d, y->n_owned, 1);
}
int bp5_vector_sadd(bp5_vector_t y, double s, double a, bp5_vector_t x) {
  int rc;
  if ((rc = same_layout(y, x))) return rc;
  BP5_CUDA(cudaSetDevice(y->ctx->device));
  return vec_axpy(y->ctx, y->d, s, a, x->d, y->n_owned, 2);
}
int bp5_vector_scale(bp5_vector_t y, bp5_vector_t x) {
  int rc;
  if ((rc = same_layout(y, x))) return rc;
  BP5_CUDA(cudaSetDevice(y->ctx->device));
  return vec_axpy(y->ctx, y->d, 1.0, 1.0, x->d, y->n_owned, 3);
}
int bp5_vector_dot_local(bp5_vector_t x, bp5_vector_t y, double *out) {
  int rc;
  if ((rc = same_layout(x, y))) return rc;
  BP5_REQUIRE(out, "null output");
  BP5_CUDA(cudaSetDevice(x->ctx->device));
  return vec_dot(x->ctx, x->d, y->d, x->n_owned, out);
}
int bp5_vector_norm_sqr_local(bp5_vector_t x, double *out) { return bp5_vector_dot_local(x, x, out); }
int bp5_vector_all_zero_local(bp5_vector_t x, int *out) {
  BP5_REQUIRE(x && out, "null argument");
  BP5_CUDA(cudaSetDevice(x->ctx->device));
  return vec_all_zero(x->ctx, x->d, x->n_owned, out);
}
int bp5_vector_zero_out_ghosts(bp5_vector_t v) {
  BP5_REQUIRE(v, "null vector");
  if (v->n_ghost == 0) return BP5_OK;
  BP5_CUDA(cudaSetDevice(v->ctx->device));
  BP5_CUDA(cudaMemsetAsync(v->d + v->n_owned, 0, sizeof(double) * v->n_ghost, v->ctx->stream));
  return BP5_OK;
}

// ------------------------------------------------------------------- solver
int bp5_cg_solve(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diag, int variant, int control,
                 double tol, int max_its, int *last_step, double *last_value, double *history, int history_len) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && x && b, "null argument");
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return cg_solve(op, x, b, diag, variant, control, tol, max_its, last_step, last_value, history, history_len);
  BP5_ABI_GUARD_END
}

int bp5_cg_solve_host(bp5_operator_t op, double *x_host, const double *b_host, int64_t n, int x0_is_zero, int variant,
                      int control, double tol, int max_its, int *last_step, double *last_value) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && x_host && b_host, "null argument");
  BP5_REQUIRE(n == op->n_owned && op->n_ghost == 0, "host solve needs a single block and n == n_dofs");
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return solve_host(op, x_host, b_host, x0_is_zero, [&](bp5_vector_t x, bp5_vector_t b) {
    return cg_solve(op, x, b, nullptr, variant, control, tol, max_its, last_step, last_value, nullptr, 0);
  });
  BP5_ABI_GUARD_END
}


// ------------------------------------------------- user-written cell functors
int bp5_operator_matrix_free_data(bp5_operator_t op, bp5_matrix_free_data_t *out) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && out, "null argument");
  BP5_REQUIRE(op->n_ghost == 0, "the generic functor path handles a single block");
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  int rc;
  if ((rc = op->hanging ? operator_generic_data_hanging(op) : operator_generic_data(op))) return rc;
  std::memset(out, 0, sizeof(*out));
  for (int sI = 0; sI < 2; ++sI)
    for (int i = 0; i < op->n * op->n; ++i) out->hanging_interpolation[sI][i] = op->hanging_interp[sI][i];
  out->q_points = op->mf_q_points;
  out->local_to_global = op->mf_l2g;
  out->inv_jacobian = op->mf_inv_jacobian;
  out->JxW = op->mf_jxw;
  out->constraint_mask = op->mf_constraint_mask;
  out->n_cells = (unsigned int)op->n_cells;
  out->padding_length = (unsigned int)op->mf_padding;
  out->n_q_points_1d = op->n;
  out->collocation = op->prob.quadrature == BP5_QUAD_GLL;
  for (int q = 0; q < op->n; ++q)
    for (int i = 0; i < op->n; ++i) {
      out->shape_values[q * op->n + i] = op->tab.B[q * op->n + i];
      out->shape_gradients[q * op->n + i] = op->tab.Dg[q * op->n + i];
      out->co_shape_gradients[q * op->n + i] = op->tab.Dt[q * op->n + i];
    }
  return BP5_OK;
  BP5_ABI_GUARD_END
}

static void fill_tables(bp5_operator_t op, bp5_matrix_free_data_t *out) {
  out->padding_length = (unsigned int)op->mf_padding;
  out->n_q_points_1d = op->n;
  out->collocation = op->prob.quadrature == BP5_QUAD_GLL;
  for (int q = 0; q < op->n; ++q)
    for (int i = 0; i < op->n; ++i) {
      out->shape_values[q * op->n + i] = op->tab.B[q * op->n + i];
      out->shape_gradients[q * op->n + i] = op->tab.Dg[q * op->n + i];
      out->co_shape_gradients[q * op->n + i] = op->tab.Dt[q * op->n + i];
    }
}

int bp5_operator_matrix_free_data_colored(bp5_operator_t op, int color, bp5_matrix_free_data_t *out) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && out, "null argument");
  BP5_REQUIRE(color >= 0 && color < 8, "colour must be 0..7");
  BP5_CONFORMING_ONLY(op);
  BP5_REQUIRE(op->n_ghost == 0, "the generic functor path handles a single block");
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  int rc;
  if ((rc = operator_generic_data_colored(op))) return rc;
  std::memset(out, 0, sizeof(*out));
  out->q_points = op->mfc_q_points[color];
  out->local_to_global = op->mfc_l2g[color];
  out->inv_jacobian = op->mfc_inv_jacobian[color];
  out->JxW = op->mfc_jxw[color];
  out->constraint_mask = op->mfc_constraint_mask[color];
  out->n_cells = (unsigned int)op->mfc_n_cells[color];
  fill_tables(op, out);
  return BP5_OK;
  BP5_ABI_GUARD_END
}

// ------------------------------------------------- partitioned meshes: halo + stepwise CG
int bp5_operator_halo_info(bp5_operator_t op, int64_t *send_count, int64_t *send_offset, int64_t *recv_count,
                           int64_t *recv_offset) {
  BP5_REQUIRE(op && send_count && send_offset && recv_count && recv_offset, "null argument");
  return halo_info(op, send_count, send_offset, recv_count, recv_offset);
}

int bp5_operator_halo_pack(bp5_operator_t op, bp5_vector_t vec, double *sendbuf_dev) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && sendbuf_dev, "null argument");
  int rc;
  if ((rc = check_vec(op, vec))) return rc;
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return halo_pack(op, vec->d, sendbuf_dev);
  BP5_ABI_GUARD_END
}

int bp5_operator_halo_unpack_add(bp5_operator_t op, bp5_vector_t vec, const double *recvbuf_dev) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && recvbuf_dev, "null argument");
  int rc;
  if ((rc = check_vec(op, vec))) return rc;
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return halo_unpack_add(op, vec->d, recvbuf_dev);
  BP5_ABI_GUARD_END
}

int bp5_cg_step_begin(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diag, int control, double tol,
                      int max_its, double res0, int history_len) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op, "null operator");
  int rc;
  if ((rc = check_vec(op, x)) || (rc = check_vec(op, b))) return rc;
  if (diag && (rc = check_vec(op, diag))) return rc;
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return cg_step_begin(op, x, b, diag, control, tol, max_its, res0, history_len);
  BP5_ABI_GUARD_END
}

int bp5_cg_step_vectors(bp5_operator_t op, bp5_vector_t *g, bp5_vector_t *d, bp5_vector_t *h) {
  BP5_REQUIRE(op && op->g, "bp5_cg_step_begin has not been called");
  if (g) *g = op->g;
  if (d) *d = op->d;
  if (h) *h = op->h;
  return BP5_OK;
}

#define BP5_STEP_GUARD()                                                              \
  BP5_REQUIRE(op && op->cg_scalars && op->cg_x, "bp5_cg_step_begin has not been called"); \
  BP5_CUDA(cudaSetDevice(op->ctx->device))

int bp5_cg_step_update(bp5_operator_t op, int iteration) {
  BP5_ABI_GUARD_BEGIN
  BP5_STEP_GUARD();
  BP5_REQUIRE(iteration >= 1, "iterations are 1-based");
  return cg_step_update(op, iteration);
  BP5_ABI_GUARD_END
}

int bp5_cg_step_apply_local(bp5_operator_t op) {
  BP5_ABI_GUARD_BEGIN
  BP5_STEP_GUARD();
  // h (zeroed by the update step) = local cells' part of A d; the caller exchanges halos around this
  return cg_step_apply_local(op);
  BP5_ABI_GUARD_END
}

int bp5_cg_step_constrained(bp5_operator_t op) {
  BP5_ABI_GUARD_BEGIN
  BP5_STEP_GUARD();
  return cg_step_constrained(op);
  BP5_ABI_GUARD_END
}

int bp5_cg_step_local_dots(bp5_operator_t op, double *sums7_dev) {
  BP5_ABI_GUARD_BEGIN
  BP5_STEP_GUARD();
  BP5_REQUIRE(sums7_dev, "null buffer");
  return cg_step_local_dots(op, sums7_dev);
  BP5_ABI_GUARD_END
}

int bp5_cg_step_scalars(bp5_operator_t op, const double *sums7_dev) {
  BP5_ABI_GUARD_BEGIN
  BP5_STEP_GUARD();
  BP5_REQUIRE(sums7_dev, "null buffer");
  return cg_step_scalars(op, sums7_dev);
  BP5_ABI_GUARD_END
}

int bp5_cg_step_poll(bp5_operator_t op, int *state, int *last_step, double *last_value) {
  BP5_ABI_GUARD_BEGIN
  BP5_STEP_GUARD();
  return cg_step_poll(op, state, last_step, last_value);
  BP5_ABI_GUARD_END
}

int bp5_cg_step_finish(bp5_operator_t op, double *history) {
  BP5_ABI_GUARD_BEGIN
  BP5_STEP_GUARD();
  return cg_step_finish(op, history);
  BP5_ABI_GUARD_END
}

// ------------------------------------------------- peer-memory transport
int bp5_peer_export(bp5_operator_t op, int rank, int world, bp5_peer_info_t *info) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && info, "null argument");
  BP5_CONFORMING_ONLY(op);
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return peer_export(op, rank, world, info);
  BP5_ABI_GUARD_END
}

int bp5_peer_connect(bp5_operator_t op, const bp5_peer_info_t *all_infos, const int32_t *upper_rank,
                     const int32_t *lower_rank) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && all_infos && upper_rank && lower_rank, "null argument");
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return peer_connect(op, all_infos, upper_rank, lower_rank);
  BP5_ABI_GUARD_END
}

int bp5_peer_vmult(bp5_operator_t op, bp5_vector_t dst, bp5_vector_t src) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op, "null operator");
  int rc;
  if ((rc = check_vec(op, dst)) || (rc = check_vec(op, src))) return rc;
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return peer_vmult(op, dst, src);
  BP5_ABI_GUARD_END
}

int bp5_peer_cg_solve(bp5_operator_t op, bp5_vector_t x, bp5_vector_t b, bp5_vector_t diag, int control, double tol,
                      int max_its, int *last_step, double *last_value, double *history, int history_len) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op, "null operator");
  int rc;
  if ((rc = check_vec(op, x)) || (rc = check_vec(op, b))) return rc;
  if (diag && (rc = check_vec(op, diag))) return rc;
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return cg_solve_peer(op, x, b, diag, control, tol, max_its, last_step, last_value, history, history_len);
  BP5_ABI_GUARD_END
}

int bp5_peer_world_size(bp5_operator_t op) { return op ? peer_world_size(op) : 1; }

int bp5_vector_update_ghost_values(bp5_operator_t op, bp5_vector_t vec) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op, "null operator");
  int rc;
  if ((rc = check_vec(op, vec))) return rc;
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  if (peer_world_size(op) == 1 && op->n_ghost == 0) return BP5_OK;     // single block: nothing to exchange
  return peer_update_ghost_values(op, vec);
  BP5_ABI_GUARD_END
}

int bp5_vector_compress_add(bp5_operator_t op, bp5_vector_t vec) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op, "null operator");
  int rc;
  if ((rc = check_vec(op, vec))) return rc;
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  if (peer_world_size(op) == 1 && op->n_ghost == 0) return BP5_OK;
  return peer_compress_add(op, vec);
  BP5_ABI_GUARD_END
}

int bp5_peer_cg_solve_host(bp5_operator_t op, double *x_host, const double *b_host, int64_t n, int x0_is_zero,
                           int control, double tol, int max_its, int *last_step, double *last_value) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && x_host && b_host, "null argument");
  BP5_REQUIRE(n == op->n_owned, "host buffers hold this block's owned range: n == n_owned");
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return solve_host(op, x_host, b_host, x0_is_zero, [&](bp5_vector_t x, bp5_vector_t b) {
    return cg_solve_peer(op, x, b, nullptr, control, tol, max_its, last_step, last_value, nullptr, 0);
  });
  BP5_ABI_GUARD_END
}

int bp5_peer_allreduce(bp5_operator_t op, double *values, int n) {
  BP5_ABI_GUARD_BEGIN
  BP5_REQUIRE(op && values && n >= 1 && n <= 8, "bad argument");
  BP5_CUDA(cudaSetDevice(op->ctx->device));
  return peer_allreduce_host(op, values, n);
  BP5_ABI_GUARD_END
}

}  // extern "C"
