"""-m gpu: the CUDA path (through the C ABI) against the oracle and the committed golden
fixtures.  Tolerance: fp64 operator application <= 1e-12 relative L2 error (north star);
CG: same iteration count +-1 to the same tolerance, solution to 1e-8."""
import json
import os

import numpy as np
import pytest

from conftest import ladder

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
TOL = 1e-12


def _dc():
    import dealceed_b200 as dc
    return dc


def _vmult(ctx, op, u):
    src, dst = op.initialize_dof_vector(), op.initialize_dof_vector()
    src.import_host(u)
    op.vmult(dst, src)
    out = dst.to_host()
    src.close(); dst.close()
    return out


def relerr(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


@pytest.mark.parametrize("p", range(1, 9))
def test_vmult_matches_golden_fixture_and_oracle(gpu_ctx, p):
    """every degree x quadrature x operator x (affine|deformed): committed fixture AND live oracle"""
    dc = _dc()
    import oracle as O
    gold = np.load(os.path.join(GOLD, "vmult_cases.npz"))
    for quad in (0, 1):
        for kind in (0, 1):
            for deform in (0, 1):
                key = f"p{p}_q{quad}_k{kind}_d{deform}"
                cells = tuple(int(c) for c in gold[key + "_cells"])
                op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, operator_kind=kind,
                                                                 deformation=deform, eps=0.1))
                u = np.random.default_rng(p).standard_normal(op.n_owned)
                got = _vmult(gpu_ctx, op, u)
                assert relerr(got, gold[key + "_out"]) <= TOL, key
                m = O.OracleMesh(p, cells, quad=quad, deform=deform, eps=0.1)
                assert relerr(got, m.vmult(u, kind=kind)) <= TOL, key
                assert np.abs(op.coefficients() - m.metric()).max() <= 1e-12 * np.abs(m.metric()).max(), key
                op.close()


@pytest.mark.parametrize("p,cells", [(2, (1, 1, 1)), (4, (1, 1, 1)), (8, (1, 1, 1)), (3, (7, 1, 1)), (2, (5, 3, 1)),
                                     (4, (3, 2, 1)), (5, (2, 2, 1)), (6, (4, 1, 1)), (7, (3, 1, 1)), (1, (33, 1, 1))])
def test_ragged_and_minimal_meshes(gpu_ctx, p, cells):
    """cell counts that do not fill the last tile, single cells, one-cell-thick slabs"""
    dc = _dc()
    import oracle as O
    for quad in (0, 1):
        op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad))
        m = O.OracleMesh(p, cells, quad=quad)
        u = np.random.default_rng(7).standard_normal(m.n_dofs)
        assert relerr(_vmult(gpu_ctx, op, u), m.vmult(u)) <= TOL
        op.close()


def test_vmult_semantics_zero_out_and_constrained_copy(gpu_ctx):
    """do_zero_out=false accumulates (bp5/step-64.cu:270-271); Dirichlet rows copy src (:275)"""
    dc = _dc()
    import oracle as O
    p, cells = 3, (3, 3, 2)
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells))
    m = O.OracleMesh(p, cells)
    rng = np.random.default_rng(3)
    u, w = rng.standard_normal(m.n_dofs), rng.standard_normal(m.n_dofs)
    src, dst = op.initialize_dof_vector(), op.initialize_dof_vector()
    src.import_host(u); dst.import_host(w)
    op.do_zero_out = False
    op.vmult(dst, src)
    got = dst.to_host()
    ref = m.vmult(u, dst=w.copy())
    assert relerr(got, ref) <= TOL
    bm = m.boundary_mask()
    assert np.array_equal(got[bm], u[bm])
    op.do_zero_out = True
    op.vmult(dst, src)
    assert relerr(dst.to_host(), m.vmult(u)) <= TOL
    # the two halves separately
    dst.set(0.0)
    op.cell_loop(dst, src)
    half = dst.to_host()
    op.copy_constrained_values(dst, src)
    assert relerr(dst.to_host(), m.vmult(u)) <= TOL and not np.array_equal(half[bm], u[bm])
    for v in (src, dst):
        v.close()
    op.close()


def test_config1_p4_32cubed(gpu_ctx):
    """BASELINE config 1 (p=4, 32^3 cells, 2,146,689 DoFs): operator and 200-iteration CG vs fixture"""
    dc = _dc()
    g = json.load(open(os.path.join(GOLD, "config1_p4_32.json")))
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(4, (32, 32, 32), upper=(1., 1., 1.)))
    assert op.n_owned == g["n_dofs"]
    n = op.n_owned
    # boundary mask from coordinates
    xyz = op.dof_coordinates()
    bm = np.any((xyz == 0.0) | (xyz == 1.0), axis=1)
    u = np.random.default_rng(4).standard_normal(n); u[bm] = 0
    v = _vmult(gpu_ctx, op, u)
    assert np.linalg.norm(v) == pytest.approx(g["vmult_seed4_l2"], rel=1e-12)
    np.testing.assert_allclose(v[:: n // 16][:16], g["vmult_seed4_sample"], rtol=1e-10, atol=1e-12 * np.abs(v).max())
    b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    assert b.l2_norm() == pytest.approx(g["b_l2"], rel=1e-12)
    ctl = dc.IterationNumberControl(200, 1e-6 * b.l2_norm())
    op.do_zero_out = False
    dc.SolverCGFullMerge(ctl).solve(op, x, b)
    assert ctl.last_step() == g["its"] == 200          # terminates at the cap (SURVEY 8d)
    np.testing.assert_allclose(ctl.history[::20], g["history_every_20"], rtol=1e-6)
    assert x.l2_norm() == pytest.approx(g["x_l2"], rel=1e-8)
    for v_ in (b, x):
        v_.close()
    op.close()


@pytest.mark.parametrize("cycle", [7, 8, 12, 13])
@pytest.mark.parametrize("quad", ["gauss", "gll"])
def test_bp5_ladder_cg_iteration_parity(gpu_ctx, cycle, quad):
    """reference mesh ladder, degree 5, tol 1e-6 (bp5/step-64.cu:443-445,724-730): merged and standard CG"""
    dc = _dc()
    g = json.load(open(os.path.join(GOLD, "bp5_ladder_p5.json")))[f"cycle{cycle}_{quad}"]
    cells, upper = ladder(cycle)
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(5, cells, quadrature=0 if quad == "gauss" else 1, upper=upper))
    assert op.n_owned == g["n_dofs"]
    b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    assert b.l2_norm() == pytest.approx(g["b_l2"], rel=1e-12)
    tol = 1e-6 * b.l2_norm()
    for Solver, key, zero in ((dc.SolverCGFullMerge, "its_merged", False), (dc.SolverCG, "its_standard", True)):
        ctl = dc.IterationNumberControl(200, tol)
        op.do_zero_out = zero
        x.set(0.0)
        Solver(ctl).solve(op, x, b)
        assert abs(ctl.last_step() - g[key]) <= 1
        assert x.l2_norm() == pytest.approx(g["x_l2"], rel=1e-6)
        if key == "its_merged" and ctl.last_step() == g[key]:
            # residual history: tight while the residual is large, loose in the last digits
            # before convergence (rounding-sensitive; the iteration count is the parity criterion)
            h, hg = np.asarray(ctl.history), np.asarray(g["history"])
            big = hg > 1e-3 * hg[0]
            np.testing.assert_allclose(h[big], hg[big], rtol=1e-6)
            np.testing.assert_allclose(h[~big], hg[~big], rtol=0.25)
    b.close(); x.close(); op.close()


@pytest.mark.parametrize("refine,its_ref,norm_ref", [(1, 27, 0.0205439), (2, 60, 0.0205269), (3, 114, 0.0205261)])
def test_step64_helmholtz_known_answers_on_gpu(gpu_ctx, refine, its_ref, norm_ref):
    """upstream deal.II step-64 tutorial output reproduced by the CUDA path (Q3, tol 1e-12|b|, SolverControl)"""
    dc = _dc()
    import oracle as O
    c = 2 ** refine
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(3, (c, c, c), operator_kind=dc.OP_HELMHOLTZ, upper=(1., 1., 1.)))
    b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    for Solver, zero in ((dc.SolverCG, True), (dc.SolverCGFullMerge, False)):
        ctl = dc.SolverControl(op.n_owned, 1e-12 * b.l2_norm())
        op.do_zero_out = zero
        x.set(0.0)
        Solver(ctl).solve(op, x, b)
        assert abs(ctl.last_step() - its_ref) <= 1
        m = O.OracleMesh(3, (c, c, c), quad=O.GAUSS, upper=(1., 1., 1.))
        assert f"{m.l2_norm(x.to_host()):.6g}" == f"{norm_ref:.6g}"
        assert f"{op.l2_norm(x):.6g}" == f"{norm_ref:.6g}"                 # the same integral on the device
        assert op.l2_norm(x) == pytest.approx(m.l2_norm(x.to_host()), rel=1e-7)    # per-cell norms are float-rounded
    b.close(); x.close(); op.close()


def test_solver_control_failure_and_diag_preconditioner(gpu_ctx):
    dc = _dc()
    import oracle as O
    p, cells = 3, (3, 2, 2)
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells))
    m = O.OracleMesh(p, cells)
    b, x, diag = op.initialize_dof_vector(), op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    op.do_zero_out = False
    ctl = dc.SolverControl(3, 0.0)
    with pytest.raises(dc.NoConvergence):
        dc.SolverCGFullMerge(ctl).solve(op, x, b)
    assert ctl.last_step() == 3
    # zero right-hand side: converged at step 0, x untouched
    z = op.initialize_dof_vector()
    ctl = dc.SolverControl(10, 0.0)
    x.set(0.0)
    dc.SolverCGFullMerge(ctl).solve(op, x, z)
    assert ctl.last_step() == 0 and x.all_zero()
    # non-trivial diagonal in the preconditioner slot (solver.h:421), non-zero start vector
    d = 1.0 / (1.0 + np.arange(m.n_dofs) % 3)
    diag.import_host(d)
    bh = b.to_host()
    tol = 1e-8 * np.linalg.norm(bh)
    x0 = np.random.default_rng(5).standard_normal(m.n_dofs); x0[m.boundary_mask()] = 0
    xo, its, *_ = m.cg(bh, x0=x0, variant=1, control=1, tol=tol, max_its=500, diag=d)
    for Solver, zero in ((dc.SolverCGFullMerge, False), (dc.SolverCG, True)):
        ctl = dc.SolverControl(500, tol)
        op.do_zero_out = zero
        x.import_host(x0)
        Solver(ctl).solve(op, x, b, preconditioner=diag)
        assert abs(ctl.last_step() - its) <= 1
        assert relerr(x.to_host(), xo) <= 1e-7
    for v in (b, x, diag, z):
        v.close()
    op.close()


def test_full_size_properties(gpu_ctx):
    """size-independent properties at a BASELINE-scale mesh (p=6, 40^3 cells, 13.9M DoFs):
    linearity, symmetry u.Av = v.Au, A*1 = 0 off the boundary, positive definiteness"""
    dc = _dc()
    p, c = 6, 40
    for quad in (0, 1):
        op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, (c, c, c), quadrature=quad, deformation=1, eps=0.1))
        n = op.n_owned
        xyz = op.dof_coordinates()
        bm = np.any((xyz == 0.0) | (xyz == float(c)), axis=1)
        rng = np.random.default_rng(11)
        u, v = rng.standard_normal(n), rng.standard_normal(n)
        u[bm] = 0; v[bm] = 0
        U, V, W, AU, AV, AW = [op.initialize_dof_vector() for _ in range(6)]
        U.import_host(u); V.import_host(v); W.import_host(2.0 * u - 3.0 * v)
        op.vmult(AU, U); op.vmult(AV, V); op.vmult(AW, W)
        uav, vau, uau = U.dot_local(AV), V.dot_local(AU), U.dot_local(AU)
        assert abs(uav - vau) <= 1e-11 * abs(uav)
        assert uau > 0
        lin = AW.to_host() - (2.0 * AU.to_host() - 3.0 * AV.to_host())
        assert np.linalg.norm(lin) <= 1e-12 * np.linalg.norm(AW.to_host())
        U.set(1.0)
        op.vmult(AU, U)
        r = AU.to_host()
        assert np.abs(r[~bm]).max() <= 1e-10 and np.all(r[bm] == 1.0)
        for t in (U, V, W, AU, AV, AW):
            t.close()
        op.close()


def test_vector_ops(gpu_ctx):
    dc = _dc()
    n = 100003
    rng = np.random.default_rng(0)
    a, b = rng.standard_normal(n), rng.standard_normal(n)
    A, B = dc.Vector(gpu_ctx, n), dc.Vector(gpu_ctx, n)
    assert A.all_zero()
    A.import_host(a); B.import_host(b)
    assert not A.all_zero()
    assert A.dot_local(B) == pytest.approx(a @ b, rel=1e-12)
    assert A.l2_norm() == pytest.approx(np.linalg.norm(a), rel=1e-13)
    A.add(2.5, B); a = a + 2.5 * b
    np.testing.assert_allclose(A.to_host(), a, rtol=1e-14, atol=1e-14)   # FMA contraction on the device
    A.sadd(0.5, -1.0, B); a = 0.5 * a - b
    np.testing.assert_allclose(A.to_host(), a, rtol=1e-14, atol=1e-14)
    A.equ(-1.0, B)
    np.testing.assert_array_equal(A.to_host(), -b)
    A.set(3.0)
    assert np.all(A.to_host() == 3.0)
    A.close(); B.close()


def test_host_buffer_solve_matches_device_solve(gpu_ctx):
    """bp5_cg_solve_host (the end-to-end entry point bench.py times): zero-start flag and explicit x0 agree with
    the device-vector solve and the oracle"""
    dc = _dc()
    import oracle as O
    p, cells = 3, (4, 3, 3)
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=dc.QUAD_GLL, deformation=1, eps=0.1))
    m = O.OracleMesh(p, cells, quad=O.GLL, deform=1, eps=0.1)
    bh = m.rhs()
    tol = 1e-8 * np.linalg.norm(bh)
    xo, its, _, _, _ = m.cg(bh, variant=1, control=1, tol=tol, max_its=500)
    op.do_zero_out = False
    for zero_flag in (True, False):
        x = np.full(op.n_owned, 123.0) if zero_flag else np.zeros(op.n_owned)   # garbage must be ignored with the flag
        ctl = dc.SolverControl(500, tol)
        dc.cg_solve_host(op, x, bh, ctl, x0_is_zero=zero_flag)
        assert abs(ctl.last_step() - its) <= 1
        assert relerr(x, xo) <= 1e-7
    # a non-zero initial guess: start from the solution, expect immediate convergence
    x = xo.copy()
    ctl = dc.SolverControl(500, 1e-6 * np.linalg.norm(bh))
    dc.cg_solve_host(op, x, bh, ctl, x0_is_zero=False)
    assert ctl.last_step() <= 1
    op.close()


@pytest.mark.parametrize("p", range(1, 9))
def test_on_the_fly_geometry_matches_stored_metric_and_oracle(gpu_ctx, p):
    """BASELINE config 5: geometry recomputed in the kernel from the nodal coordinates vs the stored metric tensor:
    both <= 1e-12 from the oracle (SURVEY 8c.3 asks 1e-13 between them on small meshes), affine and deformed cells,
    ragged tile counts; CG iteration parity"""
    dc = _dc()
    import oracle as O
    for cells, deform in (((3, 2, 2), 1), ((2, 3, 1), 0), ((1, 1, 1), 1)):
        m = O.OracleMesh(p, cells, quad=O.GLL, deform=deform, eps=0.1)
        u = np.random.default_rng(10 + p).standard_normal(m.n_dofs)
        ref = m.vmult(u)
        outs = {}
        for mode in (dc.GEOM_STORED, dc.GEOM_ON_THE_FLY):
            op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=dc.QUAD_GLL, deformation=deform, eps=0.1,
                                                             geometry_mode=mode))
            outs[mode] = _vmult(gpu_ctx, op, u)
            assert relerr(outs[mode], ref) <= TOL, (p, cells, deform, mode)
            if mode == dc.GEOM_ON_THE_FLY:
                assert "on-the-fly" in op.kernel_name
                with pytest.raises(dc.Bp5Error):
                    op.coefficients()                       # nothing stored
                b = op.initialize_dof_vector(); x = op.initialize_dof_vector()
                op.assemble_rhs(b)
                bh = b.to_host()
                tol = 1e-8 * np.linalg.norm(bh)
                ctl = dc.SolverControl(1000, tol)
                op.do_zero_out = False
                dc.SolverCGFullMerge(ctl).solve(op, x, b)
                xo, its, _, _, _ = m.cg(bh, variant=1, control=1, tol=tol, max_its=1000)
                assert abs(ctl.last_step() - its) <= 1
                if np.linalg.norm(xo) > 0:
                    assert relerr(x.to_host(), xo) <= 1e-7
                b.close(); x.close()
            op.close()
        assert relerr(outs[dc.GEOM_ON_THE_FLY], outs[dc.GEOM_STORED]) <= 1e-13


@pytest.mark.parametrize("p", range(1, 9))
@pytest.mark.parametrize("quad", [0, 1])
def test_on_the_fly_geometry_affine_fast_path(gpu_ctx, p, quad):
    """geometry on the fly on an undeformed mesh: the Jacobian is one constant diagonal, the kernel forms
    G = w_q diag(hy hz / hx, ...) from three parameters and streams no geometry at all (16 bytes per DoF).  Both
    quadratures, anisotropic cells, ragged tile counts: == stored metric to 1e-13, == oracle, CG iteration parity."""
    dc = _dc()
    import oracle as O
    cells, upper = (3, 2, 3), (1.5, 2.0, 0.75)
    m = O.OracleMesh(p, cells, quad=quad, upper=upper)
    u = np.random.default_rng(20 + p).standard_normal(m.n_dofs)
    ref = m.vmult(u)
    outs = {}
    for mode in (dc.GEOM_STORED, dc.GEOM_ON_THE_FLY):
        op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, upper=upper, geometry_mode=mode))
        outs[mode] = _vmult(gpu_ctx, op, u)
        assert relerr(outs[mode], ref) <= TOL
        if mode == dc.GEOM_ON_THE_FLY:
            assert "affine" in op.kernel_name
            assert op.algorithmic_bytes()[0] == 16.0 * op.n_owned
            b = op.initialize_dof_vector(); x = op.initialize_dof_vector()
            op.assemble_rhs(b)
            bh = b.to_host()
            tol = 1e-8 * np.linalg.norm(bh)
            ctl = dc.SolverControl(1000, tol)
            op.do_zero_out = False
            dc.SolverCGFullMerge(ctl).solve(op, x, b)
            xo, its, _, _, _ = m.cg(bh, variant=1, control=1, tol=tol, max_its=1000)
            assert abs(ctl.last_step() - its) <= 1
            assert relerr(x.to_host(), xo) <= 1e-7
            b.close(); x.close()
        op.close()
    assert relerr(outs[dc.GEOM_ON_THE_FLY], outs[dc.GEOM_STORED]) <= 1e-13


@pytest.mark.parametrize("p", range(1, 9))
@pytest.mark.parametrize("quad,kind", [(0, 0), (0, 1), (1, 1)])
def test_on_the_fly_geometry_general_kernel(gpu_ctx, p, quad, kind):
    """geometry on the fly for the reference's default quadrature QGauss(p+1) (bp5/step-64.cu:243-247) and for the
    Helmholtz operator (step-64/step-64.cu:201-219, coefficient a(x) evaluated at the recomputed quadrature
    points): the CTA rebuilds the tile's coefficient in shared memory from the nodal coordinates.  Deformed and
    affine (anisotropic) meshes, ragged tile counts, a single cell: == stored metric to 1e-13, == oracle, dst += A src,
    merged-CG iteration parity (fused d.Ad path)."""
    dc = _dc()
    import oracle as O
    for cells, deform, upper in (((3, 2, 2), 1, None), ((2, 3, 1), 0, (1.5, 2.0, 0.75)), ((1, 1, 1), 1, None)):
        if deform == 0 and kind == 0:
            continue                                    # Poisson on affine meshes: the constant-Jacobian fast path
        m = O.OracleMesh(p, cells, quad=quad, deform=deform, eps=0.1, upper=upper)
        u = np.random.default_rng(30 + p).standard_normal(m.n_dofs)
        ref = m.vmult(u, kind=kind)
        outs = {}
        for mode in (dc.GEOM_STORED, dc.GEOM_ON_THE_FLY):
            op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, operator_kind=kind, deformation=deform,
                                                             eps=0.1, upper=upper, geometry_mode=mode))
            outs[mode] = _vmult(gpu_ctx, op, u)
            assert relerr(outs[mode], ref) <= TOL, (p, cells, deform, mode)
            if mode == dc.GEOM_ON_THE_FLY:
                assert "bp5_apply_otfg_kernel" in op.kernel_name and "on-the-fly" in op.kernel_name
                assert op.algorithmic_bytes()[0] == 16.0 * op.n_owned + 24.0 * op.n_owned
                with pytest.raises(dc.Bp5Error):
                    op.coefficients()                       # nothing stored
                # dst += A src (do_zero_out = false, bp5/step-64.cu:270-271)
                src, dst = op.initialize_dof_vector(), op.initialize_dof_vector()
                w = np.random.default_rng(40 + p).standard_normal(m.n_dofs)
                src.import_host(u); dst.import_host(w)
                op.do_zero_out = False
                op.vmult(dst, src)
                assert relerr(dst.to_host(), m.vmult(u, kind=kind, dst=w.copy())) <= TOL
                src.close(); dst.close()
                b = op.initialize_dof_vector(); x = op.initialize_dof_vector()
                op.assemble_rhs(b)
                bh = b.to_host()
                if np.linalg.norm(bh) > 0:
                    tol = 1e-8 * np.linalg.norm(bh)
                    ctl = dc.SolverControl(1000, tol)
                    dc.SolverCGFullMerge(ctl).solve(op, x, b)
                    xo, its, _, _, _ = m.cg(bh, kind=kind, variant=1, control=1, tol=tol, max_its=1000)
                    assert abs(ctl.last_step() - its) <= 1
                    assert relerr(x.to_host(), xo) <= 1e-7
                b.close(); x.close()
            op.close()
        # (interpolation to the Gauss points, then the collocation derivative: one more rounding stage than the
        # stored metric's direct derivative matrix)
        assert relerr(outs[dc.GEOM_ON_THE_FLY], outs[dc.GEOM_STORED]) <= 2e-13


def test_on_the_fly_geometry_rejects_refined_meshes(gpu_ctx):
    dc = _dc()
    with pytest.raises(dc.Bp5Error):
        dc.PoissonOperator(gpu_ctx, dc.make_problem(3, (4, 4, 4), geometry_mode=dc.GEOM_ON_THE_FLY, quadrature=1,
                                                     refine_lo=(0, 0, 0), refine_hi=(2, 2, 2)))


@pytest.mark.parametrize("p,quad,kind", [(2, 0, 0), (3, 1, 0), (4, 0, 1), (5, 1, 0)])
def test_diagonal_and_jacobi_preconditioner(gpu_ctx, p, quad, kind):
    """bp5_operator_compute_diagonal against the dense numpy assembly; Jacobi-preconditioned merged CG against the
    oracle's preconditioned CG (the diag slot of solver.h:421 with something other than ones, SURVEY 8f.2)"""
    dc = _dc()
    import oracle as O
    import bp5_numpy as NP
    cells = (2, 2, 1) if p > 3 else (3, 2, 2)
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, operator_kind=kind, deformation=1, eps=0.1))
    A = NP.NumpyBP5(p, cells, quad="gll" if quad else "gauss", deform=1, eps=0.1).assemble(helmholtz=bool(kind), apply_bc=True)
    dref = np.asarray(A.diagonal() if hasattr(A, "diagonal") else np.diag(A)).ravel()
    d = op.initialize_dof_vector()
    op.compute_diagonal(d)
    assert relerr(d.to_host(), dref) <= 1e-12
    op.compute_diagonal(d, invert=True)
    assert relerr(d.to_host(), 1.0 / dref) <= 1e-12
    m = O.OracleMesh(p, cells, quad=quad, deform=1, eps=0.1)
    b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    bh = b.to_host()
    tol = 1e-9 * np.linalg.norm(bh)
    ctl = dc.SolverControl(2000, tol)
    op.do_zero_out = False
    dc.SolverCGFullMerge(ctl).solve(op, x, b, preconditioner=d)
    xo, its, _, _, ok = m.cg(bh, kind=kind, variant=1, control=1, tol=tol, max_its=2000, diag=1.0 / dref)
    assert ok and abs(ctl.last_step() - its) <= 1
    assert relerr(x.to_host(), xo) <= 1e-7
    for v in (d, b, x):
        v.close()
    op.close()


def test_l2_norm_on_deformed_mesh(gpu_ctx):
    dc = _dc()
    import oracle as O
    for p, quad in ((2, 0), (4, 1), (7, 0)):
        cells = (3, 2, 2) if p < 7 else (2, 1, 1)
        op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, deformation=1, eps=0.1))
        m = O.OracleMesh(p, cells, quad=quad, deform=1, eps=0.1)
        u = np.random.default_rng(p).standard_normal(m.n_dofs)
        v = op.initialize_dof_vector()
        v.import_host(u)
        assert op.l2_norm(v) == pytest.approx(m.l2_norm(u), rel=1e-7)    # Vector<float> cellwise_norm, bp5/step-64.cu:603
        v.close(); op.close()


@pytest.mark.parametrize("variant", ["merged", "standard"])
def test_nan_residual_is_reported_as_no_convergence(gpu_ctx, variant):
    """A non-finite right-hand side makes alpha and the residual estimate NaN.  The reference's sqrt(NaN) fails
    SolverControl::check and solve() throws NoConvergence (bp5/solver.h:504-507,539); a clamp that swallowed the
    NaN would report success with a garbage x."""
    dc = _dc()
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(3, (3, 3, 2), quadrature=1))
    b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
    op.assemble_rhs(b)
    bh = b.to_host()
    bh[op.n_owned // 2] = np.inf
    b.import_host(bh)
    op.do_zero_out = False
    solver = dc.SolverCGFullMerge if variant == "merged" else dc.SolverCG
    for control in (dc.IterationNumberControl(50, 1e-6), dc.SolverControl(50, 1e-6)):
        x.set(0.0)
        with pytest.raises(dc.NoConvergence):
            solver(control).solve(op, x, b)
        assert control.last_step() < 50 and not np.isfinite(control.last_value())
    b.close(); x.close(); op.close()


@pytest.mark.parametrize("p,cells", [(1, (9, 8, 7)), (2, (5, 4, 3)), (4, (5, 5, 3)), (5, (4, 3, 3)), (6, (5, 3, 2)),
                                     (7, (3, 3, 2)), (8, (3, 2, 1)), (3, (1, 1, 1))])
@pytest.mark.parametrize("quad", [0, 1])
def test_colored_cell_order_is_bitwise_reproducible(gpu_ctx, p, cells, quad):
    """cell_order = COLORED (MatrixFree's use_coloring = true; bp5/step-64.cu:243 sets false): eight colour passes of
    the tuned kernel with plain adds.  Same operator as the atomic path and the oracle (1e-12), and -- what the
    atomics cannot give -- the same bits on every run, for vmult and for the whole merged-CG history.
    Cell counts are odd/ragged so that colours have different sizes and partly filled tiles."""
    dc = _dc()
    import oracle as O
    for kind in (0, 1):
        m = O.OracleMesh(p, cells, quad=quad, deform=1, eps=0.1)
        u = np.random.default_rng(11 * p + kind).standard_normal(m.n_dofs)
        ref = m.vmult(u, kind=kind)
        op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=quad, operator_kind=kind, deformation=1,
                                                         eps=0.1, cell_order=dc.CELL_ORDER_COLORED))
        assert np.abs(op.coefficients() - m.metric()).max() <= 1e-12 * np.abs(m.metric()).max()
        outs = [_vmult(gpu_ctx, op, u) for _ in range(3)]
        assert relerr(outs[0], ref) <= TOL
        assert all(np.array_equal(outs[0], o) for o in outs[1:])
        b, x = op.initialize_dof_vector(), op.initialize_dof_vector()
        op.assemble_rhs(b)
        op.do_zero_out = False
        runs = []
        for _ in range(2):
            ctl = dc.SolverControl(300, 1e-8 * b.l2_norm())
            x.set(0.0)
            dc.SolverCGFullMerge(ctl).solve(op, x, b)
            runs.append((ctl.last_step(), np.asarray(ctl.history).copy(), x.to_host()))
        assert runs[0][0] == runs[1][0]
        assert np.array_equal(runs[0][1], runs[1][1]) and np.array_equal(runs[0][2], runs[1][2])
        xo, its, _, _, _ = m.cg(m.rhs(), kind=kind, variant=1, control=1, tol=1e-8 * np.linalg.norm(m.rhs()), max_its=300)
        assert abs(runs[0][0] - its) <= 1
        assert relerr(runs[0][2], xo) <= 1e-6
        b.close(); x.close(); op.close()


def test_colored_cell_order_rejects_partitions_and_on_the_fly_geometry(gpu_ctx):
    dc = _dc()
    for kw in (dict(part_grid=(2, 1, 1)), dict(geometry_mode=dc.GEOM_ON_THE_FLY, quadrature=1)):
        with pytest.raises(dc.Bp5Error) as e:
            dc.PoissonOperator(gpu_ctx, dc.make_problem(3, (4, 4, 4), cell_order=dc.CELL_ORDER_COLORED, **kw))
        assert "coloured cell order" in str(e.value)
