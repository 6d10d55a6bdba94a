"""-m gpu: the cell kernels' steady-state tile loop against the CPU oracle.

Every cell kernel is a persistent loop, `for (tile = tile_begin + blockIdx.x; tile < n_tiles; tile += gridDim.x)`, and
most of its pipelining only runs from a CTA's second tile on: the metric of the next tile is fetched behind the
current one, cell descriptors are loaded two tiles ahead and gathered values one tile ahead (at p = 8 with
Gauss-Lobatto, copied into shared memory with cp.async), and the fused d.Ad partial sums over all of a CTA's tiles.
On the small meshes of the other tests every CTA runs at most one tile, so none of that code runs there.

The meshes here are sized so that every CTA runs at least three tiles, and every case asserts that premise from an
upper bound of the grid (`_assert_tiles_per_cta`): the grid is at most blocks-per-SM x SMs, and blocks-per-SM is at
most 32 (the hardware's limit) and at most 2048 // NT (threads per SM over threads per CTA) where NT is known.  The
meshes are deformed, so that every cell has its own metric (a kernel that used another tile's metric would pass on
an undeformed mesh), and their cell counts leave the last tile partly filled wherever a tile holds more than one
cell."""
import math
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
TOL = 1e-12
MAX_CTAS_PER_SM = 32          # resident CTAs per SM on sm_100, whatever the kernel
MAX_THREADS_PER_SM = 2048
COLOR_GRID_CAP = 512          # kApplyPartialCap / 8: the grid of one colour's launch in the coloured cell order

# cells per mesh, stored metric and default cell order: >= 3 x the grid bound in tiles on 148 SMs, n_cells % cpt != 0
STORED = {1: (63, 61, 60), 2: (47, 46, 46), 3: (39, 39, 38), 4: (34, 33, 32), 5: (28, 28, 28), 6: (26, 25, 25),
          7: (25, 25, 23), 8: (23, 21, 20)}
# geometry on the fly: one mesh per degree for the stored-metric, bp5_apply_otf, bp5_apply_otfg and affine kernels
OTF = {2: (60, 59, 57), 4: (33, 33, 33), 5: (35, 35, 35), 8: (26, 24, 23)}
# coloured cell order: every colour holds >= 3 x 512 tiles
COLORED = {1: (74, 74, 72), 4: (42, 41, 39), 8: (24, 24, 22)}


def _dc():
    import dealceed_b200 as dc
    return dc


@pytest.fixture(scope="module")
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _cells_per_tile(op):
    return int(re.search(r"cells_per_tile=(\d+)", op.kernel_name).group(1))


def _grid_bound(op, sm_count):
    """An upper bound of the cell kernel's grid.  For the stored-metric kernels (and the affine on-the-fly path, which
    is the same kernel) the CTA has NT = ceil(cpt (p+1)^2 / 32) * 32 threads (ApplyCfg::NT); for the others NT is not
    known here and only the hardware's limit of CTAs per SM is used."""
    per_sm = MAX_CTAS_PER_SM
    if op.kernel_name.startswith("bp5_apply_kernel<"):
        nt = math.ceil(_cells_per_tile(op) * (op.problem.degree + 1) ** 2 / 32) * 32
        per_sm = min(per_sm, MAX_THREADS_PER_SM // nt)
    return per_sm * sm_count


def _assert_tiles_per_cta(op, sm_count, ragged=True):
    """every CTA of the default cell order's launch runs >= 3 tiles; returns cells per tile"""
    cpt = _cells_per_tile(op)
    n_tiles = -(-op.n_cells // cpt)
    bound = _grid_bound(op, sm_count)
    assert n_tiles >= 3 * bound, f"{op.kernel_name}: {n_tiles} tiles for up to {bound} CTAs"
    if ragged:
        assert cpt == 1 or op.n_cells % cpt != 0, f"{op.kernel_name}: {op.n_cells} cells fill every tile"
    return cpt


def _color_tiles(cells, cpt):
    """tiles of each colour of the coloured cell order (colour = parity of the three cell indices, each colour padded
    to whole tiles; see operator_plan_tiles)"""
    out = []
    for c in range(8):
        cnt = 1
        for d in range(3):
            cnt *= cells[d] // 2 if (c >> d) & 1 else (cells[d] + 1) // 2
        out.append(-(-cnt // cpt))
    return out


def _vmult(op, u, w=None):
    """op.vmult(dst, src) with src = u and dst = w on entry (garbage the overwriting kernel must not keep)"""
    src, dst = op.initialize_dof_vector(), op.initialize_dof_vector()
    src.import_host(u)
    dst.import_host(np.full_like(u, 1e300) if w is None else w)
    op.vmult(dst, src)
    out = dst.to_host()
    src.close(); dst.close()
    return out


def relerr(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _compare(got, ref, mesh, what, cpt=None, tol=TOL):
    """<= tol relative L2 error and <= tol max|ref| in the max norm.  On failure, name the first cell with a bad DoF
    and, for the default cell order (processing order = lexicographic cell order), its tile: the tile's CTA is
    tile mod grid.  A wrong cell spoils the DoFs it shares with its neighbours, so the first bad cell can be a
    neighbour of the first wrong one."""
    import oracle as O
    err = np.abs(got - ref)
    rel, bound = relerr(got, ref), tol * np.abs(ref).max()
    if rel <= tol and err.max() <= bound:
        return
    cell_err = err[O._cell_dofs(mesh)].max(axis=1)
    bad = np.flatnonzero(cell_err > bound)
    c = int(bad[0]) if bad.size else int(np.argmax(cell_err))
    nx, ny, _ = mesh.cells
    where = f"cell {c} = ({c % nx}, {c // nx % ny}, {c // (nx * ny)}) of {mesh.cells}"
    if cpt is not None:
        where += f", tile {c // cpt}"
    pytest.fail(f"{what}: rel L2 error {rel:.3e}, max error {err.max():.3e} (bound {bound:.3e}); {bad.size} cells "
                f"beyond the bound, first bad {where}")


@pytest.mark.parametrize("quad", [0, 1])
@pytest.mark.parametrize("p", sorted(STORED))
def test_stored_metric_tile_loop_matches_oracle(gpu_ctx, sm_count, p, quad):
    """stored metric, default cell order, Poisson and Helmholtz: vmult (overwriting kernel), dst += A src (accumulating
    kernel, through vmult and through the bare cell loop) and the right-hand side"""
    dc = _dc()
    import oracle as O
    cells = STORED[p]
    m = O.OracleMesh(p, cells, quad=quad, deform=1, eps=0.1)
    rng = np.random.default_rng(100 + 10 * p + quad)
    u, w = rng.standard_normal(m.n_dofs), rng.standard_normal(m.n_dofs)
    for kind in (0, 1):
        op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, operator_kind=kind, deformation=1,
                                                         eps=0.1))
        assert op.kernel_name.startswith("bp5_apply_kernel<") and "metric=tma-smem" in op.kernel_name
        cpt = _assert_tiles_per_cta(op, sm_count)
        case = f"p={p} quad={quad} kind={kind}"
        _compare(_vmult(op, u), m.vmult(u, kind=kind), m, f"vmult {case}", cpt)
        op.do_zero_out = False
        _compare(_vmult(op, u, w), m.vmult(u, kind=kind, dst=w.copy()), m, f"vmult dst += A src {case}", cpt)
        src, dst = op.initialize_dof_vector(), op.initialize_dof_vector()
        src.import_host(u); dst.import_host(w)
        op.cell_loop(dst, src)
        _compare(dst.to_host(), m.vmult(u, kind=kind, semantics=2, dst=w.copy()), m, f"cell_loop {case}", cpt)
        if kind == 0:                                   # the right-hand side does not depend on the operator
            op.assemble_rhs(dst)
            assert relerr(dst.to_host(), m.rhs()) <= TOL, case
        src.close(); dst.close(); op.close()


# Deviation from the oracle after 30 iterations from x = 0, measured on one B200 (1000 W power limit) over the 8 cases
# below, merged / standard CG:
#   history, max_k |h_k - h_k^oracle| / h_k^oracle: worst 2.6e-12 / 8.1e-12 (p = 1, GLL), all others <= 3.6e-13;
#   solution, relative L2:                          worst 1.4e-9 / 7.4e-10 (p = 1, GLL), all others <= 7.9e-14.
# At p = 1 with Gauss-Lobatto points CG amplifies rounding differences far more than elsewhere: the oracle's own
# merged and standard CG differ there by 9.8e-10 in x and 5.4e-12 in the history.  The solution bound stays at 1e-8
# all the same.  A wrong d.Ad from any tile changes alpha and moves both by orders of magnitude more.
CG_HIST_TOL = 1e-9
CG_X_TOL = 1e-8


@pytest.mark.parametrize("quad", [0, 1])
@pytest.mark.parametrize("p", [1, 4, 6, 8])
def test_fused_dot_product_cg_matches_oracle(gpu_ctx, sm_count, p, quad):
    """both CG variants take d.Ad from the cell kernel's per-CTA partial sums, each summed over all of the CTA's
    tiles.  30 iterations: the first ones enqueued directly, then replayed CUDA-graph batches."""
    dc = _dc()
    import oracle as O
    cells = STORED[p]
    m = O.OracleMesh(p, cells, quad=quad, deform=1, eps=0.1)
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, deformation=1, eps=0.1))
    _assert_tiles_per_cta(op, sm_count)
    b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)                                 # == m.rhs() (test_stored_metric_tile_loop_matches_oracle)
    bh = b.to_host()
    for Solver, variant, zero in ((dc.SolverCGFullMerge, 1, False), (dc.SolverCG, 0, True)):
        ctl = dc.IterationNumberControl(30, 0.0)
        op.do_zero_out = zero
        x.set(0.0)
        Solver(ctl).solve(op, x, b)
        xo, its, _, hist, _ = m.cg(bh, variant=variant, control=0, tol=0.0, max_its=30)
        assert ctl.last_step() == its == 30
        dh = float(np.max(np.abs(ctl.history - hist) / hist))
        dx = float(relerr(x.to_host(), xo))
        print(f"cg deviation p={p} quad={quad} variant={variant}: history {dh:.3e} x {dx:.3e}")
        assert dh <= CG_HIST_TOL and dx <= CG_X_TOL, (Solver.__name__, dh, dx)
    b.close(); x.close(); op.close()


@pytest.mark.parametrize("quad,kind,kernel", [(1, 0, None), (0, 0, "bp5_apply_otfg_kernel"),
                                              (1, 1, "bp5_apply_otfg_kernel")])
@pytest.mark.parametrize("p", sorted(OTF))
def test_on_the_fly_geometry_tile_loop_matches_oracle(gpu_ctx, sm_count, p, quad, kind, kernel):
    """geometry recomputed in the kernel on a deformed mesh: collocation + Poisson through bp5_apply_otf_kernel up to
    p = 4 and bp5_apply_otfg_kernel above it; Gauss and Helmholtz through bp5_apply_otfg_kernel.  == oracle to 1e-12,
    == the stored metric on the same mesh to the bounds of the small-mesh tests"""
    dc = _dc()
    import oracle as O
    cells = OTF[p]
    kernel = kernel or ("bp5_apply_otf_kernel" if p <= 4 else "bp5_apply_otfg_kernel")
    m = O.OracleMesh(p, cells, quad=quad, deform=1, eps=0.1)
    u = np.random.default_rng(200 + 10 * p + 2 * quad + kind).standard_normal(m.n_dofs)
    ref = m.vmult(u, kind=kind)
    outs = {}
    for mode in (dc.GEOM_STORED, dc.GEOM_ON_THE_FLY):
        op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, operator_kind=kind, deformation=1,
                                                         eps=0.1, geometry_mode=mode))
        if mode == dc.GEOM_ON_THE_FLY:
            assert op.kernel_name.startswith(kernel + "<") and "on-the-fly" in op.kernel_name, op.kernel_name
        cpt = _assert_tiles_per_cta(op, sm_count)
        outs[mode] = _vmult(op, u)
        _compare(outs[mode], ref, m, f"vmult p={p} quad={quad} kind={kind} {op.kernel_name}", cpt)
        op.close()
    # the general kernel interpolates to the Gauss points, then takes the collocation derivative: one more rounding
    # stage than the stored metric's direct derivative matrix
    bound = 1e-13 if kernel == "bp5_apply_otf_kernel" else 2e-13
    assert relerr(outs[dc.GEOM_ON_THE_FLY], outs[dc.GEOM_STORED]) <= bound


@pytest.mark.parametrize("quad", [0, 1])
@pytest.mark.parametrize("p", sorted(OTF))
def test_affine_on_the_fly_tile_loop_matches_oracle(gpu_ctx, sm_count, p, quad):
    """geometry on the fly on an undeformed mesh of anisotropic cells: the Jacobian is one constant diagonal formed
    from kernel parameters.  == oracle to 1e-12, == the stored metric to 1e-13"""
    dc = _dc()
    import oracle as O
    cells = OTF[p]
    upper = (0.5 * cells[0], 1.0 * cells[1], 0.25 * cells[2])
    m = O.OracleMesh(p, cells, quad=quad, upper=upper)
    u = np.random.default_rng(300 + 10 * p + quad).standard_normal(m.n_dofs)
    ref = m.vmult(u)
    outs = {}
    for mode in (dc.GEOM_STORED, dc.GEOM_ON_THE_FLY):
        op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, upper=upper, geometry_mode=mode))
        if mode == dc.GEOM_ON_THE_FLY:
            assert "affine" in op.kernel_name, op.kernel_name
        cpt = _assert_tiles_per_cta(op, sm_count)
        outs[mode] = _vmult(op, u)
        _compare(outs[mode], ref, m, f"vmult p={p} quad={quad} {op.kernel_name}", cpt)
        op.close()
    assert relerr(outs[dc.GEOM_ON_THE_FLY], outs[dc.GEOM_STORED]) <= 1e-13


@pytest.mark.parametrize("quad", [0, 1])
@pytest.mark.parametrize("p", sorted(COLORED))
def test_colored_tile_loop_matches_oracle_and_repeats_bitwise(gpu_ctx, p, quad):
    """coloured cell order: one launch per colour, each with at most 512 CTAs; every colour holds >= 3 x 512 tiles.
    == oracle to 1e-12; the same bits on a second run, for vmult and for a 30-iteration merged-CG history"""
    dc = _dc()
    import oracle as O
    cells = COLORED[p]
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, deformation=1, eps=0.1,
                                                     cell_order=dc.CELL_ORDER_COLORED))
    tiles = _color_tiles(cells, _cells_per_tile(op))
    assert min(tiles) >= 3 * COLOR_GRID_CAP, tiles
    m = O.OracleMesh(p, cells, quad=quad, deform=1, eps=0.1)
    u = np.random.default_rng(400 + 10 * p + quad).standard_normal(m.n_dofs)
    outs = [_vmult(op, u) for _ in range(2)]
    _compare(outs[0], m.vmult(u), m, f"coloured vmult p={p} quad={quad}")
    assert np.array_equal(outs[0], outs[1])
    b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    op.do_zero_out = False
    runs = []
    for _ in range(2):
        ctl = dc.IterationNumberControl(30, 0.0)
        x.set(0.0)
        dc.SolverCGFullMerge(ctl).solve(op, x, b)
        assert ctl.last_step() == 30
        runs.append((np.asarray(ctl.history).copy(), x.to_host()))
    assert np.array_equal(runs[0][0], runs[1][0]) and np.array_equal(runs[0][1], runs[1][1])
    b.close(); x.close(); op.close()


def test_vector_ops_with_several_grid_stride_passes(gpu_ctx):
    """n > blocks x threads of every vector kernel (the reductions run 592 x 256 threads), so each thread loops over
    several elements; n is odd, so the last pass is partial.  Reductions against exactly rounded sums: the bound is
    a worst-case rounding bound (< 300 additions per result) relative to the sum of the terms' magnitudes."""
    dc = _dc()
    n = 2 ** 25 + 7
    rng = np.random.default_rng(12)
    a, b = rng.standard_normal(n), rng.standard_normal(n)
    A, B = dc.Vector(gpu_ctx, n), dc.Vector(gpu_ctx, n)
    A.import_host(a); B.import_host(b)
    ab, aa = a * b, a * a
    assert abs(A.dot_local(B) - math.fsum(ab)) <= 1e-13 * np.abs(ab).sum()
    assert abs(A.l2_norm() ** 2 - math.fsum(aa)) <= 1e-13 * aa.sum()
    A.add(2.5, B); a = a + 2.5 * b
    np.testing.assert_allclose(A.to_host(), a, rtol=1e-14, atol=1e-14)   # FMA contraction on the device
    A.sadd(0.5, -1.0, B); a = 0.5 * a - b
    np.testing.assert_allclose(A.to_host(), a, rtol=1e-14, atol=1e-14)
    A.equ(-1.5, B)
    np.testing.assert_array_equal(A.to_host(), -1.5 * b)
    # all_zero must reach the last element
    z = np.zeros(n)
    z[-1] = 1e-300
    A.import_host(z)
    assert not A.all_zero()
    z[-1] = 0.0
    A.import_host(z)
    assert A.all_zero()
    A.close(); B.close()
