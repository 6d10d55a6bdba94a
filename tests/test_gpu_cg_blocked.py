"""-m gpu: the merged CG in its blocked layout.

On one conforming block in the default cell order, bp5_cg_solve runs the merged CG with its work vectors in a layout of
its own, [interior blocks | skeleton] (BlockedLayout in csrc/common.h): every cell's interior DoFs are one contiguous
block, the skeleton comes in three classes (z-face planes, y-face planes, x-face planes only).  b, x and the Jacobi
diagonal are permuted in at the start of a solve and x back at the end; users only ever see the lexicographic layout.

The layout is taken where the iteration's working set (five vectors and the metric) exceeds the L2 cache -- only there
is there DRAM traffic for it to save -- so the meshes here have 1.7-3.8 M DoFs; odd-shaped boxes give every degree
cells of every kind and every skeleton class both lower and upper faces.

References: the stepwise API (bp5_cg_step_*), which runs the same iteration in the lexicographic layout -- the two may
differ only in the order of the sums -- and the CPU oracle."""


def _box(p, n=122):
    """about 1.8 M DoFs at degree p, three different cell counts"""
    c = n // p
    return (c + 1, c, c - 1)
import ctypes as C
import math
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _dc():
    import dealceed_b200 as dc
    return dc


def relerr(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _stepwise_solve(dc, op, x, b, diag, control):
    """the merged CG over the stepwise ABI (lexicographic layout); x must be zero"""
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
    sums.close()
    hist[0] = res0
    return its.value, hist[: its.value + 1], x.to_host()


# Two CGs that differ only in the order of their sums drift apart once rounding is amplified (late iterations, high
# degree: 1e-11 to 1e-6 relative in the histories of converged solves, now and then one iteration more).  So the first
# FIXED_ITS iterations are compared tightly: to 1e-12 against the stepwise API (the same iteration, other sum order),
# to 1e-10 against the oracle (another implementation).  Converged solves (|r| <= 1e-10 |b|) are compared by their
# iteration count and their solution: two solutions that both meet that residual differ by up to cond(A) 1e-10.
FIXED_ITS = 12      # > 3 warm-up iterations + one 8-iteration CUDA-graph batch: the replayed path is covered
STEPWISE, ORACLE, SOLUTION = 1e-12, 1e-10, 1e-7


def _merged(dc, op, b, pre, control, x0=None):
    x = op.initialize_dof_vector()
    if x0 is not None:
        x.import_host(x0)
    op.do_zero_out = False
    dc.SolverCGFullMerge(control).solve(op, x, b, preconditioner=pre)
    out = (control.last_step(), np.asarray(control.history), x.to_host())
    x.close()
    return out


def _check_against_stepwise(dc, op, jacobi):
    b, x, diag = op.initialize_dof_vector(), op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    pre = None
    if jacobi:
        op.compute_diagonal(diag, invert=True)
        pre = diag
    tiny, tol = 1e-30 * b.l2_norm(), 1e-10 * b.l2_norm()
    its, hist, xm = _merged(dc, op, b, pre, dc.IterationNumberControl(FIXED_ITS, tiny))
    x.set(0.0)
    its_s, hist_s, xs = _stepwise_solve(dc, op, x, b, pre, dc.IterationNumberControl(FIXED_ITS, tiny))
    assert its == its_s == FIXED_ITS
    assert relerr(hist, hist_s) <= STEPWISE
    assert relerr(xm, xs) <= STEPWISE
    its, _, xm = _merged(dc, op, b, pre, dc.SolverControl(5000, tol))
    x.set(0.0)
    its_s, _, xs = _stepwise_solve(dc, op, x, b, pre, dc.SolverControl(5000, tol))
    assert abs(its - its_s) <= 1
    assert relerr(xm, xs) <= SOLUTION
    for v in (b, x, diag):
        v.close()


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("quad", [0, 1])
def test_blocked_merged_cg_matches_the_stepwise_api(gpu_ctx, p, quad):
    """every degree on an odd box: the layout map and its two permutations, every column class of the cell kernel"""
    dc = _dc()
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, _box(p), quadrature=quad, deformation=1, eps=0.1))
    for jacobi in (False, True):
        _check_against_stepwise(dc, op, jacobi)
    op.close()


@pytest.mark.parametrize("kind,geom", [(1, 0), (0, 1)])
def test_helmholtz_and_affine_fast_path_take_the_blocked_path_and_agree(gpu_ctx, kind, geom):
    """Helmholtz (7 metric planes) and the affine on-the-fly kernel have blocked instantiations too (the diagonal, and
    with it Jacobi, needs the stored metric)"""
    dc = _dc()
    pr = dc.make_problem(5, (32, 31, 30) if geom else _box(5), quadrature=1, operator_kind=kind,
                         geometry_mode=dc.GEOM_ON_THE_FLY if geom else dc.GEOM_STORED, deformation=0 if geom else 1,
                         eps=0.1)
    op = dc.PoissonOperator(gpu_ctx, pr)
    for jacobi in ((False,) if geom else (False, True)):
        _check_against_stepwise(dc, op, jacobi)
    op.close()


@pytest.mark.parametrize("quad", [0, 1])
@pytest.mark.parametrize("deform", [0, 1])
@pytest.mark.parametrize("jacobi", [False, True])
def test_blocked_merged_cg_matches_the_oracle(gpu_ctx, quad, deform, jacobi):
    dc = _dc()
    import oracle as O
    p, cells = 4, _box(4)
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, deformation=deform, eps=0.1))
    m = O.OracleMesh(p, cells, quad=quad, deform=deform, eps=0.1)
    b, d = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    op.compute_diagonal(d, invert=True)
    pre, dh = (d, d.to_host()) if jacobi else (None, None)
    bh = b.to_host()
    tiny = 1e-30 * np.linalg.norm(bh)
    its, hist, x = _merged(dc, op, b, pre, dc.IterationNumberControl(FIXED_ITS, tiny))
    xo, its_o, _, hist_o, _ = m.cg(bh, variant=1, control=0, tol=tiny, max_its=FIXED_ITS, diag=dh)
    assert its == its_o == FIXED_ITS
    assert relerr(hist, hist_o) <= ORACLE
    assert relerr(x, xo) <= ORACLE
    for v in (b, d):
        v.close()
    op.close()


@pytest.mark.parametrize("jacobi", [False, True])
def test_blocked_merged_cg_from_a_nonzero_start(gpu_ctx, jacobi):
    """x != 0: g = A x - b in the user's layout, then g and x permuted; x comes back in the user's layout"""
    dc = _dc()
    import oracle as O
    p, cells = 3, _box(3)
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, deformation=1, eps=0.1))
    m = O.OracleMesh(p, cells, deform=1, eps=0.1)
    b, x, d = op.initialize_dof_vector(), op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    op.compute_diagonal(d, invert=True)
    bh = b.to_host()
    x0 = np.random.default_rng(3).standard_normal(m.n_dofs) * 1e-3
    x0[m.boundary_mask()] = 0.0
    x.import_host(x0)
    ctl = dc.IterationNumberControl(FIXED_ITS, 1e-30 * np.linalg.norm(bh))
    op.do_zero_out = False
    dc.SolverCGFullMerge(ctl).solve(op, x, b, preconditioner=d if jacobi else None)
    xo, its, _, hist, _ = m.cg(bh, x0=x0, variant=1, control=0, tol=ctl.tol, max_its=FIXED_ITS,
                               diag=d.to_host() if jacobi else None)
    assert ctl.last_step() == its == FIXED_ITS
    assert relerr(np.asarray(ctl.history), hist) <= ORACLE
    assert relerr(x.to_host(), xo) <= ORACLE
    for v in (b, x, d):
        v.close()
    op.close()


@pytest.mark.parametrize("p,cells,quad", [(6, (26, 25, 25), 1), (2, (47, 46, 46), 0)])
def test_blocked_merged_cg_where_every_cta_loops_over_several_tiles(gpu_ctx, p, cells, quad):
    """the cell kernel's pipeline (descriptors two tiles ahead, values one tile ahead) over the blocked layout"""
    dc = _dc()
    import torch
    import oracle as O
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, deformation=1, eps=0.05))
    cpt = int(re.search(r"cells_per_tile=(\d+)", op.kernel_name).group(1))
    nt = math.ceil(cpt * (p + 1) ** 2 / 32) * 32
    grid_bound = min(32, 2048 // nt) * torch.cuda.get_device_properties(0).multi_processor_count
    assert math.prod(cells) / cpt >= 2 * grid_bound
    m = O.OracleMesh(p, cells, quad=quad, deform=1, eps=0.05)
    b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    bh = b.to_host()
    its_max = 24
    ctl = dc.IterationNumberControl(its_max, 1e-14 * np.linalg.norm(bh))
    op.do_zero_out = False
    dc.SolverCGFullMerge(ctl).solve(op, x, b)
    xo, its, _, hist, _ = m.cg(bh, variant=1, control=0, tol=ctl.tol, max_its=its_max)
    assert ctl.last_step() == its == its_max
    assert relerr(np.asarray(ctl.history), hist) <= 1e-10
    assert relerr(x.to_host(), xo) <= 1e-10
    for v in (b, x):
        v.close()
    op.close()


def _kernels_of_one_solve(dc, op, x, b, pre, solver=None):
    """names of the kernels one merged-CG solve runs (torch.profiler)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    op.do_zero_out = False
    ctl = dc.IterationNumberControl(FIXED_ITS, 0.0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        (solver or dc.SolverCGFullMerge)(ctl).solve(op, x, b, preconditioner=pre)
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type.name == "CUDA"]


@pytest.mark.parametrize("case", ["poisson", "jacobi", "x0", "helmholtz", "affine", "colored", "standard", "small"])
def test_the_blocked_path_is_taken_where_it_applies(gpu_ctx, case):
    """permutations in (b; x when non-zero; the diagonal with Jacobi) and out (x), and the cell kernel's blocked
    instantiation (its last template argument) in every iteration; none of it for the coloured cell order, the
    standard CG and a mesh whose working set fits in L2"""
    dc = _dc()
    kw = dict(quadrature=1, deformation=1, eps=0.1)
    if case == "helmholtz":
        kw["operator_kind"] = dc.OP_HELMHOLTZ
    if case == "affine":
        kw = dict(quadrature=1, geometry_mode=dc.GEOM_ON_THE_FLY)
    if case == "colored":
        kw["cell_order"] = dc.CELL_ORDER_COLORED
    cells = (5, 4, 3) if case == "small" else (40, 39, 38) if case == "affine" else _box(4)
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(4, cells, **kw))
    b, x, d = op.initialize_dof_vector(), op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    pre = None
    if case == "jacobi":
        op.compute_diagonal(d, invert=True)
        pre = d
    if case == "x0":
        x.import_host(np.random.default_rng(4).standard_normal(op.n_owned) * 1e-3)
    names = _kernels_of_one_solve(dc, op, x, b, pre, dc.SolverCG if case == "standard" else None)
    permutes = sum("blocked_permute_kernel" in n for n in names)
    blocked_cells = sum("bp5_apply_kernel<" in n and n.split(">")[0].endswith("true") for n in names)
    if case in ("colored", "standard", "small"):
        assert permutes == 0 and blocked_cells == 0
    else:
        assert permutes == {"jacobi": 3, "x0": 3}.get(case, 2)
        assert blocked_cells == FIXED_ITS
    for v in (b, x, d):
        v.close()
    op.close()
