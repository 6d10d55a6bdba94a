"""-m gpu: the single-block merged CG (bp5_cg_solve) and the stepwise API (bp5_cg_step_*, what a partitioned mesh
drives around its own halo exchange) run the same iteration: the same update, cell-loop, Dirichlet-copy and
dot-product kernels with the same partial sums; only where the scalar recurrences run differs (fused into the dots
kernel, or a separate kernel after the caller's allreduce).  Under the coloured cell order, which has no atomics,
both must give the same bits."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _dc():
    import dealceed_b200 as dc
    return dc


def _stepwise_solve(dc, op, x, b, diag, control):
    """SolverCGFullMerge over the stepwise ABI, as DistributedPoisson.cg_solve drives it, with no halo to exchange"""
    B = dc.bindings
    lib = B.lib()
    res0 = b.l2_norm()
    hist_len = control.max_its + 2
    sums = dc.Vector(op.ctx, 8)
    B._check(lib.bp5_cg_step_begin(op.h, x.h, b.h, diag.h if diag is not None else None, control.kind, control.tol,
                                   control.max_its, res0, hist_len))
    st, its, res = C.c_int(0), C.c_int(0), C.c_double(0.0)
    for it in range(1, control.max_its + 1):
        B._check(lib.bp5_cg_step_update(op.h, it))
        B._check(lib.bp5_cg_step_apply_local(op.h))
        B._check(lib.bp5_cg_step_constrained(op.h))
        B._check(lib.bp5_cg_step_local_dots(op.h, sums.get_values()))
        B._check(lib.bp5_cg_step_scalars(op.h, sums.get_values()))
        B._check(lib.bp5_cg_step_poll(op.h, C.byref(st), C.byref(its), C.byref(res)))
        if st.value != 0:
            break
    hist = np.full(hist_len, np.nan)
    B._check(lib.bp5_cg_step_finish(op.h, hist.ctypes.data_as(B._dp)))
    B._check(lib.bp5_cg_step_poll(op.h, C.byref(st), C.byref(its), C.byref(res)))
    sums.close()
    hist[0] = res0
    return st.value, its.value, hist[: its.value + 1], x.to_host()


@pytest.mark.parametrize("p,cells", [(2, (5, 4, 3)), (5, (3, 3, 2)), (8, (2, 2, 1))])
@pytest.mark.parametrize("quad", [0, 1])
@pytest.mark.parametrize("jacobi", [False, True])
def test_merged_solve_and_stepwise_api_give_the_same_bits(gpu_ctx, p, cells, quad, jacobi):
    dc = _dc()
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, deformation=1, eps=0.1,
                                                     cell_order=dc.CELL_ORDER_COLORED))
    b, x, diag = op.initialize_dof_vector(), op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    op.compute_diagonal(diag, invert=True)
    pre = diag if jacobi else None
    tol = 1e-10 * b.l2_norm()

    merged = dc.SolverControl(2000, tol)
    dc.SolverCGFullMerge(merged).solve(op, x, b, preconditioner=pre)
    x_merged = x.to_host()

    x.set(0.0)
    state, its, hist, x_step = _stepwise_solve(dc, op, x, b, pre, dc.SolverControl(2000, tol))

    assert state == 1
    assert its == merged.last_step() and its > 11    # bp5_cg_solve replayed at least one CUDA-graph batch
    assert np.array_equal(hist, merged.history)
    assert np.array_equal(x_step, x_merged)
    for v in (b, x, diag):
        v.close()
    op.close()
