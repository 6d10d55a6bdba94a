"""Geometric multigrid on the B200 (csrc/mg.cu) against the numpy reference (oracle/mg_numpy.py): transfer, eigenvalue
estimate, smoother and V-cycle vectors, MG-preconditioned CG solves, status codes and rejections."""
import functools

import numpy as np
import pytest

from mg_numpy import NumpyMG, prolongation

pytestmark = pytest.mark.gpu

QUADS = {"gauss": 0, "gll": 1}


def _dc():
    import dealceed_b200 as dc
    return dc


def _vec(op, arr=None):
    v = op.initialize_dof_vector()
    if arr is not None:
        v.import_host(arr)
    return v


def _interior_random(rng, op):
    u = rng.standard_normal(op.n_owned)
    m = op.dof_coordinates()
    lo, hi = np.array(op.problem.lower), np.array(op.problem.upper)
    bnd = np.any(np.isclose(m, lo) | np.isclose(m, hi), axis=1)
    u[bnd] = 0.0
    return u


@functools.lru_cache(maxsize=None)
def _numpy_levels(p, cells, quad, helmholtz, deform, max_levels):
    """assembled reference levels (expensive at high p); lambdas are overwritten per test"""
    return NumpyMG(p, cells, quad=quad, helmholtz=helmholtz, deform=deform, eps=0.1 if deform else 0.0,
                   max_levels=max_levels, coarse_tol=1e-14, lambdas={l: 1.0 for l in range(1, 8)})


# ---------------------------------------------------------------- 1. transfer
@pytest.mark.parametrize("p", range(1, 9))
def test_transfer_matches_numpy_and_is_adjoint_and_repeatable(gpu_ctx, p):
    dc = _dc()
    cells = (4, 2, 2)
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells))
    mg = dc.Multigrid(op, max_levels=2)
    assert mg.n_levels == 2
    cop = mg.level_operator(0)
    P = prolongation(p, (2, 1, 1))
    assert P.shape == (op.n_owned, cop.n_owned)
    rng = np.random.default_rng(p)
    uc, uf = rng.standard_normal(cop.n_owned), rng.standard_normal(op.n_owned)
    src_c, dst_f, src_f, dst_c = _vec(cop, uc), _vec(op), _vec(op, uf), _vec(cop)
    mg.prolongate(1, dst_f, src_c)
    got, want = dst_f.to_host(), P @ uc
    assert np.linalg.norm(got - want) <= 1e-13 * np.linalg.norm(want)
    mg.restrict(1, dst_c, src_f)
    gotr, wantr = dst_c.to_host(), P.T @ uf
    bc = _interior_random(rng, cop) == 0.0
    wantr[bc] = 0.0
    assert np.linalg.norm(gotr - wantr) <= 1e-13 * np.linalg.norm(wantr)
    # bitwise repeatable
    again_f, again_c = _vec(op), _vec(cop)
    mg.prolongate(1, again_f, src_c)
    mg.restrict(1, again_c, src_f)
    assert np.array_equal(again_f.to_host(), got) and np.array_equal(again_c.to_host(), gotr)
    # <P u, v> = <u, R v> on interior vectors
    ui, vi = _interior_random(rng, cop), _interior_random(rng, op)
    src_c.import_host(ui); src_f.import_host(vi)
    mg.prolongate(1, dst_f, src_c)
    mg.restrict(1, dst_c, src_f)
    lhs, rhs = dst_f.to_host() @ vi, ui @ dst_c.to_host()
    assert abs(lhs - rhs) <= 1e-13 * np.linalg.norm(dst_f.to_host()) * np.linalg.norm(vi)
    # a degree-p polynomial sampled on the coarse nodes is reproduced at the fine nodes
    poly = lambda X: (X[:, 0] ** min(p, 2)) * (1.0 + X[:, 1]) ** max(p - 2, 0) + X[:, 2]
    src_c.import_host(poly(cop.dof_coordinates()))
    mg.prolongate(1, dst_f, src_c)
    want = poly(op.dof_coordinates())
    assert np.max(np.abs(dst_f.to_host() - want)) <= 1e-12 * np.max(np.abs(want))
    for v in (src_c, dst_f, src_f, dst_c, again_f, again_c):
        v.close()
    mg.close(); op.close()


# ---------------------------------------------------------------- 2. eigenvalue estimate
@pytest.mark.parametrize("quad", ["gauss", "gll"])
@pytest.mark.parametrize("p,cells", [(2, (4, 4, 4)), (4, (4, 4, 2)), (6, (2, 2, 2))])
def test_eigenvalue_estimate_brackets_the_exact_value(gpu_ctx, p, cells, quad):
    dc = _dc()
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=QUADS[quad]))
    mg = dc.Multigrid(op)
    ref = _numpy_levels(p, cells, quad, False, 0, 0)
    assert mg.n_levels == ref.n_levels
    for l in range(1, mg.n_levels):
        lam, exact = mg.lambda_max(l), ref.exact_lambda(l)
        assert 0.9 * exact <= lam <= (1.0 + 1e-10) * exact, (l, lam, exact)
    mg.close(); op.close()


# ---------------------------------------------------------------- 3. smoother and V-cycle vectors
_CASES = [(p, q, h, dfm) for p in (1, 2, 4, 6) for q in ("gauss", "gll") for h in (False, True) for dfm in (0, 1)]
_CASES += [(8, "gauss", False, 0), (8, "gll", True, 1)]   # p = 8: the reference assembly takes ~30 s per mesh
_MESH = {1: (4, 4, 4), 2: (4, 4, 4), 4: (4, 4, 2), 6: (2, 2, 2), 8: (2, 2, 2)}


@pytest.mark.parametrize("p,quad,helmholtz,deform", _CASES)
def test_smoother_and_vcycle_match_numpy(gpu_ctx, p, quad, helmholtz, deform):
    dc = _dc()
    cells = _MESH[p]
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=QUADS[quad],
                                                     operator_kind=int(helmholtz), deformation=deform,
                                                     eps=0.1 if deform else 0.0))
    mg = dc.Multigrid(op, coarse_tol=1e-14)
    ref = _numpy_levels(p, cells, quad, helmholtz, deform, 0)
    assert mg.n_levels == ref.n_levels >= 2
    for l in range(1, mg.n_levels):
        ref.lam[l] = mg.lambda_max(l)
    # p = 8: NumpyBP5's 1D tables come from the monomial route and its assembled matrix agrees with the C++ oracle
    # to 1.3e-11 only (one Chebyshev smoothing of the two references differs by 1.1e-11): the reference sets the bound
    tol = 1e-12 if p < 8 else 5e-11
    rng = np.random.default_rng(7)
    top = mg.n_levels - 1
    b = _interior_random(rng, op)
    bv, xv = _vec(op, b), _vec(op)
    mg.smooth(top, xv, bv)
    want = ref.smooth(top, None, b)
    assert np.linalg.norm(xv.to_host() - want) <= tol * np.linalg.norm(want)
    # from a non-zero x
    x0 = _interior_random(rng, op)
    xv.import_host(x0)
    mg.smooth(top, xv, bv)
    want = ref.smooth(top, x0, b)
    assert np.linalg.norm(xv.to_host() - want) <= tol * np.linalg.norm(want)
    mg.vmult(xv, bv)
    want = ref.vcycle(b)
    assert np.linalg.norm(xv.to_host() - want) <= 1e-10 * np.linalg.norm(want)
    bv.close(); xv.close(); mg.close(); op.close()


# ---------------------------------------------------------------- 4. solves
def _mg_solve(dc, op, tol_rel, mg=None, control=None, **params):
    own = mg is None
    mg = mg or dc.Multigrid(op, **params)
    b, x = _vec(op), _vec(op)
    op.assemble_rhs(b)
    ctl = control or dc.SolverControl(100, tol_rel * b.l2_norm())
    dc.SolverCG(ctl).solve(op, x, b, preconditioner=mg)
    out = x.to_host(), ctl.last_step(), ctl.history, b.l2_norm(), op.l2_norm(x)
    b.close(); x.close()
    if own:
        mg.close()
    return out


def test_mg_solution_equals_jacobi_solution(gpu_ctx):
    dc = _dc()
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(4, (8, 8, 8)))
    x_mg, its, hist, bn, _ = _mg_solve(dc, op, 1e-10)
    assert its <= 10 and hist[-1] <= 1e-10 * bn
    assert np.all(hist[1:] <= 2.0 * hist[:-1]), hist
    b, x, diag = _vec(op), _vec(op), _vec(op)
    op.assemble_rhs(b)
    op.compute_diagonal(diag, invert=True)
    dc.SolverCG(dc.SolverControl(5000, 1e-13 * b.l2_norm())).solve(op, x, b, preconditioner=diag)
    xj = x.to_host()
    assert np.linalg.norm(x_mg - xj) <= 1e-8 * np.linalg.norm(xj)
    b.close(); x.close(); diag.close(); op.close()


@pytest.mark.parametrize("p,cells,quad,helmholtz,deform", [
    (2, (16, 16, 16), "gll", 0, 0), (2, (16, 16, 16), "gauss", 0, 0),
    (4, (8, 8, 8), "gll", 0, 0), (4, (8, 8, 8), "gauss", 0, 0),
    (6, (8, 8, 8), "gll", 0, 0), (6, (8, 8, 8), "gauss", 0, 0),
    (4, (8, 8, 8), "gauss", 1, 0), (4, (8, 8, 8), "gauss", 0, 1)])
def test_mg_iteration_counts(gpu_ctx, p, cells, quad, helmholtz, deform):
    dc = _dc()
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=QUADS[quad], operator_kind=helmholtz,
                                                     deformation=deform, eps=0.1 if deform else 0.0))
    _, its, hist, bn, _ = _mg_solve(dc, op, 1e-10)
    assert its <= 10, its
    op.close()


@pytest.mark.parametrize("p,ladder", [(4, (8, 16, 32)), (6, (4, 8, 16))])
def test_mg_iteration_counts_are_h_independent(gpu_ctx, p, ladder):
    dc = _dc()
    counts = []
    for c in ladder:
        op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, (c, c, c), quadrature=dc.QUAD_GLL))
        counts.append(_mg_solve(dc, op, 1e-10)[1])
        op.close()
    print("MG-CG iterations", p, ladder, counts)
    assert counts[-1] <= counts[0] + 2, counts
    assert max(counts) <= 10, counts


def test_config2_helmholtz_norm_with_far_fewer_iterations(gpu_ctx):
    """config 2: step-64 Helmholtz, p = 4, 64^3 cells (16.97 M DoFs), 1e-12|b|: plain CG needs 1356 iterations"""
    dc = _dc()
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(4, (64, 64, 64), operator_kind=dc.OP_HELMHOLTZ,
                                                     upper=(1., 1., 1.)))
    _, its, hist, bn, norm = _mg_solve(dc, op, 1e-12)
    print(f"config 2 MG-CG: {its} iterations, |u|_L2 = {norm:.7g}")
    assert f"{norm:.6g}" == "0.0205261"
    assert its <= 30, its
    op.close()


# ---------------------------------------------------------------- 5. status codes and rejections
def test_controls_nan_and_zero_rhs(gpu_ctx):
    dc = _dc()
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(3, (4, 4, 4)))
    mg = dc.Multigrid(op)
    ctl = dc.IterationNumberControl(2, 1e-14)
    _mg_solve(dc, op, 0.0, mg=mg, control=ctl)
    assert ctl.last_step() == 2
    with pytest.raises(dc.NoConvergence):
        _mg_solve(dc, op, 0.0, mg=mg, control=dc.SolverControl(2, 1e-14))
    b, x = _vec(op), _vec(op)
    op.assemble_rhs(b)
    bh = b.to_host()
    bh[len(bh) // 2] = np.nan
    b.import_host(bh)
    ctl = dc.SolverControl(20, 1e-10)
    with pytest.raises(dc.NoConvergence):
        dc.SolverCG(ctl).solve(op, x, b, preconditioner=mg)
    b.set(0.0); x.set(0.0)
    ctl = dc.SolverControl(20, 1e-10)
    dc.SolverCG(ctl).solve(op, x, b, preconditioner=mg)
    assert ctl.last_step() == 0 and x.all_zero()
    with pytest.raises(dc.Bp5Error) as e:
        dc.SolverCGFullMerge(ctl).solve(op, x, b, preconditioner=mg)
    assert e.value.code == dc.bindings.ERR_UNSUPPORTED
    b.close(); x.close(); mg.close(); op.close()


@pytest.mark.parametrize("kw", [dict(part_grid=(2, 1, 1)), dict(refine_lo=(1, 1, 1), refine_hi=(2, 2, 2)),
                                dict(geometry_mode=1), dict(cell_order=1)])
def test_unsupported_operators(gpu_ctx, kw):
    dc = _dc()
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(2, (4, 4, 4), **kw))
    with pytest.raises(dc.Bp5Error) as e:
        dc.Multigrid(op)
    assert e.value.code == dc.bindings.ERR_UNSUPPORTED
    op.close()


def test_odd_mesh_has_one_level_and_solves(gpu_ctx):
    dc = _dc()
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(3, (3, 4, 4)))
    mg = dc.Multigrid(op)
    assert mg.n_levels == 1
    with pytest.raises(dc.Bp5Error):
        mg.lambda_max(0)
    x, its, hist, bn, _ = _mg_solve(dc, op, 1e-10, mg=mg)
    assert hist[-1] <= 1e-10 * bn and its <= 5
    mg.close(); op.close()


# ---------------------------------------------------------------- 6. C++ facade
def test_cpp_multigrid_driver():
    """examples/bp5_mg.cc (plain g++ on the facade): the multigrid solve reproduces the Jacobi solve's ||u||_L2 to 1e-8
    in at most 10 iterations, for BP5 and the step-64 Helmholtz operator"""
    import os
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.check_call(["make", "-C", os.path.join(root, "examples")], stdout=subprocess.DEVNULL)
    out = subprocess.run([os.path.join(root, "build", "examples", "bp5_mg"), "--degree", "4", "--cells", "16"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    print(out.stdout)
    solved = re.findall(r"(jacobi|multigrid).*Solved in (\d+) iterations.*solution norm: (\S+)", out.stdout)
    assert [s[0] for s in solved] == ["jacobi", "multigrid"] * 2, out.stdout
    for (_, its_j, norm_j), (_, its_mg, norm_mg) in zip(solved[::2], solved[1::2]):
        assert int(its_mg) <= 10 < int(its_j)
        assert float(norm_mg) == pytest.approx(float(norm_j), rel=1e-8)
