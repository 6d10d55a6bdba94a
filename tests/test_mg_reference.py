"""CPU checks of the numpy multigrid reference (oracle/mg_numpy.py) and of the Python Multigrid class's argument
checks: the reference is what the GPU multigrid is compared against, so its transfer must be exact nodal
interpolation, its V-cycle a symmetric positive definite preconditioner, and its iteration counts independent of h."""
import numpy as np
import pytest

from bp5_numpy import lobatto01
from mg_numpy import NumpyMG, level_cells, prolongation


def lattice_coords(p, cells, h):
    """1D node coordinates of the lattice along each direction for cell size h"""
    xi, _ = lobatto01(p + 1)
    out = []
    for c, hd in zip(cells, h):
        pts = np.concatenate([(k + xi[:-1]) * hd for k in range(c)] + [[c * hd]])
        out.append(pts)
    return out


@pytest.mark.parametrize("p", [1, 2, 3, 4, 6, 8])
def test_prolongation_reproduces_polynomials_of_degree_p(p):
    coarse = (2, 1, 3)
    fine = tuple(2 * c for c in coarse)
    P = prolongation(p, coarse)
    xc = lattice_coords(p, coarse, (1.0, 1.0, 1.0))
    xf = lattice_coords(p, fine, (0.5, 0.5, 0.5))
    rng = np.random.default_rng(p)
    for _ in range(3):
        e = rng.integers(0, p + 1, size=3)
        while e.sum() > p:
            e[rng.integers(0, 3)] -= 1
        e = np.maximum(e, 0)
        poly = lambda X: (1.0 + X[0] ** e[0]) * X[1] ** e[1] * (0.5 - X[2]) ** e[2]
        Zc, Yc, Xc = np.meshgrid(xc[2], xc[1], xc[0], indexing="ij")
        Zf, Yf, Xf = np.meshgrid(xf[2], xf[1], xf[0], indexing="ij")
        got = P @ poly((Xc.ravel(), Yc.ravel(), Zc.ravel()))
        want = poly((Xf.ravel(), Yf.ravel(), Zf.ravel()))
        assert np.max(np.abs(got - want)) <= 1e-13 * max(1.0, np.max(np.abs(want))), (p, e)


def test_level_cells_halve_while_even():
    assert level_cells((8, 4, 4)) == [(2, 1, 1), (4, 2, 2), (8, 4, 4)]
    assert level_cells((6, 6, 6)) == [(3, 3, 3), (6, 6, 6)]
    assert level_cells((5, 4, 4)) == [(5, 4, 4)]
    assert level_cells((16, 16, 16), max_levels=2) == [(8, 8, 8), (16, 16, 16)]


@pytest.mark.parametrize("quad,helmholtz,deform", [("gauss", False, 0), ("gll", True, 1)])
def test_vcycle_is_symmetric_and_positive(quad, helmholtz, deform):
    mg = NumpyMG(2, (4, 4, 2), quad=quad, helmholtz=helmholtz, deform=deform, eps=0.1)
    rng = np.random.default_rng(3)
    bm = mg.bmask[-1]
    for _ in range(3):
        u, v = rng.standard_normal((2, bm.size))
        u[bm] = 0.0
        v[bm] = 0.0
        Mu, Mv = mg.vcycle(u), mg.vcycle(v)
        assert abs(u @ Mv - v @ Mu) <= 1e-13 * (u @ Mu), (u @ Mv, v @ Mu)
        assert u @ Mu > 0.0 and v @ Mv > 0.0


@pytest.mark.parametrize("p,ladder", [(2, [(4, 4, 4), (8, 8, 8)]), (4, [(2, 2, 2), (4, 4, 4)])])
def test_mg_pcg_iteration_counts_do_not_grow(p, ladder):
    counts = []
    for cells in ladder:
        mg = NumpyMG(p, cells)
        b = mg.meshes[-1].rhs()
        x, its, hist = mg.solve(b, 1e-10 * np.linalg.norm(b), max_its=50)
        assert hist[-1] <= 1e-10 * np.linalg.norm(b)
        assert np.linalg.norm(mg.A[-1] @ x - b) <= 1e-9 * np.linalg.norm(b)
        counts.append(its)
    assert max(counts) <= 8, counts
    assert counts[-1] <= counts[0], counts


# ---- argument checks of dealceed_b200.Multigrid that run before any device call
def test_multigrid_rejects_bad_parameters():
    import dealceed_b200 as dc
    with pytest.raises(TypeError, match="unknown multigrid parameter"):
        dc.Multigrid(None, smoothing_dgree=3)
    with pytest.raises(ValueError, match="non-negative integer"):
        dc.Multigrid(None, smoothing_degree=-1)
    with pytest.raises(ValueError, match="non-negative integer"):
        dc.Multigrid(None, max_levels=2.5)
    with pytest.raises(ValueError, match="non-negative number"):
        dc.Multigrid(None, coarse_tol=float("nan"))
    with pytest.raises(ValueError, match="exceed 1"):
        dc.Multigrid(None, smoothing_range=0.5)
    with pytest.raises(TypeError, match="PoissonOperator"):
        dc.Multigrid(None, smoothing_degree=4)


def test_merged_cg_rejects_a_multigrid_preconditioner():
    import dealceed_b200 as dc
    mg = dc.Multigrid.__new__(dc.Multigrid)   # no device object needed: the check precedes any library call
    with pytest.raises(dc.Bp5Error) as e:
        dc.SolverCGFullMerge(dc.SolverControl(10, 1e-8)).solve(None, None, None, preconditioner=mg)
    assert e.value.code == dc.bindings.ERR_UNSUPPORTED


def test_params_struct_matches_header():
    import ctypes
    import dealceed_b200 as dc
    assert ctypes.sizeof(dc.bindings.MgParams) == 4 + 4 + 8 + 4 + 4 + 8 + 16


def test_facade_rejects_merged_cg_with_multigrid_at_compile_time(tmp_path):
    """SolverCGFullMerge takes a DiagonalMatrix only: handing it the multigrid preconditioner does not compile, and
    SolverCG with it does (syntax check, no GPU needed)"""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    body = ('#include "dealii_b200/dealii_b200.h"\nusing namespace dealii;\n'
            'using V = LinearAlgebra::distributed::Vector<double, MemorySpace::CUDA>;\n'
            'void f(BP5::PoissonOperator<3, 2> &A, V &x, const V &b) {\n'
            '  b200::MultigridPreconditioner<3, 2, BP5_OP_POISSON> mg(A);\n  SolverControl c(10, 1e-8);\n'
            '  SOLVER<V>(c).solve(A, x, b, mg);\n}\n')
    results = {}
    for solver in ("SolverCG", "SolverCGFullMerge"):
        src = tmp_path / f"{solver}.cc"
        src.write_text(body.replace("SOLVER", solver))
        out = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(root, "include"), str(src)],
                             capture_output=True, text=True)
        results[solver] = out
    assert results["SolverCG"].returncode == 0, results["SolverCG"].stderr[-2000:]
    assert results["SolverCGFullMerge"].returncode != 0
    assert "DiagonalMatrix preconditioner only" in results["SolverCGFullMerge"].stderr
