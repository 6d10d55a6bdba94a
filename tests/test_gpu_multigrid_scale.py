"""-m gpu: the multigrid preconditioner (csrc/mg.cu) against the matrix-free reference (oracle/mg_matfree.py) on deep,
anisotropic, deformed hierarchies of 2.4-2.7 M DoFs, where every thread of the transfer, Chebyshev and random-fill
kernels runs its grid-stride loop at least twice.

Every MG launch is capped by mg_grid at 16 blocks per SM of 256 threads, G = 16 x SMs x 256 threads.  Each at-scale
case asserts its own premises (`_assert_premises`): the finest level has >= 3 G DoFs, the lattice written by the
first restriction pass (fine x, fine y, coarse z) has >= 2 G points, there are >= 3 levels, and the coarsest level
has interior DoFs, so its CG solves something.  Per case: the inverse diagonal of every level, prolongation and
restriction between every pair of levels, the eigenvalue estimate of every smoothed level against a replica of
estimate_lambda, the Chebyshev smoother from zero and from a non-zero x, the V-cycle through every level, and the
MG-preconditioned CG from a non-zero initial guess.  Smaller cases sweep the smoother parameters and compare the
diagonal for every degree."""
import numpy as np
import pytest

import oracle as O
from mg_matfree import MatfreeMG, metric_diagonal, probe_diagonal

pytestmark = pytest.mark.gpu

QUADS = {"gauss": 0, "gll": 1}
MG_BLOCKS_PER_SM, MG_THREADS = 16, 256     # mg_grid: at most 16 x SMs blocks of 256 threads
EPS = 0.1                                  # deformation of every mesh here

# bounds (relative; see the commit that added this file for the values measured on a B200)
TOL_DIAG = 1e-12        # max norm, inverse diagonal: up to 729 q-point terms per cell, summed in order
TOL_TRANSFER = 1e-13    # max norm, prolongation / restriction
TOL_LAMBDA = 1e-12      # eigenvalue estimate against the replica
TOL_SMOOTH = 1e-12      # L2, Chebyshev smoother
TOL_VCYCLE = 1e-12      # L2, V-cycle (the GPU's coarse CG stops at 1e-14 |b|, the reference's at 1e-15 |b|)
TOL_HIST = 1e-10        # residual history of the MG-CG
TOL_X = 1e-12           # solution of the MG-CG

# (p, quadrature, Helmholtz, finest cells): 193 x 129 x 97 lattices (193 x 145 x 97 at p = 6)
SCALE = [(1, "gauss", False, (192, 128, 96)), (2, "gll", False, (96, 64, 48)), (4, "gauss", True, (48, 32, 24)),
         (6, "gll", False, (32, 24, 16)), (8, "gll", False, (24, 16, 12))]


def _dc():
    import dealceed_b200 as dc
    return dc


@pytest.fixture(scope="module")
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _vec(op, arr=None):
    v = op.initialize_dof_vector()
    if arr is not None:
        v.import_host(arr)
    return v


def _host(v):
    out = v.to_host()
    v.close()
    return out


def _interior(rng, mask):
    u = rng.standard_normal(mask.size)
    u[mask] = 0.0
    return u


def _rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def _relmax(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def _assert_premises(mg, ref, sm_count):
    G = MG_BLOCKS_PER_SM * sm_count * MG_THREADS
    fine, coarse = ref.meshes[-1].nd, ref.meshes[-2].nd
    assert mg.n_levels == ref.n_levels >= 3, ref.cells
    assert mg.op.n_owned == ref.n(ref.n_levels - 1) >= 3 * G, (ref.n(ref.n_levels - 1), G)
    assert fine[0] * fine[1] * coarse[2] >= 2 * G, (fine, coarse, G)
    assert np.any(~ref.bmask[0]), ref.cells[0]


class Case:
    """one at-scale hierarchy: the GPU operator and multigrid, the reference, and what the checks share"""

    def __init__(self, gpu_ctx, sm_count, p, quad, helmholtz, cells):
        dc = _dc()
        self.name = f"p={p} {quad} {'Helmholtz' if helmholtz else 'Poisson'} {cells}"
        self.op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=QUADS[quad],
                                                              operator_kind=int(helmholtz), deformation=1, eps=EPS))
        self.mg = dc.Multigrid(self.op, coarse_tol=1e-14)
        self.ref = MatfreeMG(p, cells, quad=quad, helmholtz=helmholtz, deform=1, eps=EPS)
        _assert_premises(self.mg, self.ref, sm_count)
        self.gpu_lambda = {l: self.mg.lambda_max(l) for l in range(1, self.mg.n_levels)}
        self.replica_lambda = {l: self.ref.estimate_lambda(l) for l in range(1, self.ref.n_levels)}
        self.ref.lam = dict(self.gpu_lambda)     # smoother and V-cycle: compare with the GPU's lambda

    def close(self):
        self.mg.close()
        self.op.close()


@pytest.fixture(scope="module", params=SCALE, ids=[f"p{c[0]}-{c[1]}-{'helm' if c[2] else 'poisson'}" for c in SCALE])
def case(request, gpu_ctx, sm_count):
    c = Case(gpu_ctx, sm_count, *request.param)
    yield c
    c.close()


def test_scale_diagonal(case):
    worst = 0.0
    for l in range(case.mg.n_levels):
        lop = case.mg.level_operator(l)
        d = _vec(lop)
        lop.compute_diagonal(d, invert=True)
        err = _relmax(_host(d), case.ref.dinv[l])
        worst = max(worst, err)
        assert err <= TOL_DIAG, (case.name, l, err)
    print(f"{case.name}: inverse diagonal worst {worst:.2e}")


def test_scale_transfer(case):
    mg, ref = case.mg, case.ref
    rng = np.random.default_rng(11)
    worst = 0.0
    top = mg.n_levels - 1
    for l in range(1, mg.n_levels):
        fop, cop = mg.level_operator(l), mg.level_operator(l - 1)
        uc, uf = rng.standard_normal(cop.n_owned), rng.standard_normal(fop.n_owned)
        src_c, dst_f, src_f, dst_c = _vec(cop, uc), _vec(fop), _vec(fop, uf), _vec(cop)
        mg.prolongate(l, dst_f, src_c)
        mg.restrict(l, dst_c, src_f)
        got_p, got_r = dst_f.to_host(), dst_c.to_host()
        ep, er = _relmax(got_p, ref.prolongate(l, uc)), _relmax(got_r, ref.restrict(l, uf))
        worst = max(worst, ep, er)
        assert ep <= TOL_TRANSFER and er <= TOL_TRANSFER, (case.name, l, ep, er)
        if l == top:
            # bitwise repeatable
            mg.prolongate(l, dst_f, src_c)
            mg.restrict(l, dst_c, src_f)
            assert np.array_equal(dst_f.to_host(), got_p) and np.array_equal(dst_c.to_host(), got_r)
            # <P u, v> = <u, R v> on interior vectors
            ui, vi = _interior(rng, ref.bmask[l - 1]), _interior(rng, ref.bmask[l])
            src_c.import_host(ui)
            src_f.import_host(vi)
            mg.prolongate(l, dst_f, src_c)
            mg.restrict(l, dst_c, src_f)
            Pu, Rv = dst_f.to_host(), dst_c.to_host()
            assert abs(Pu @ vi - ui @ Rv) <= 1e-13 * np.linalg.norm(Pu) * np.linalg.norm(vi)
        for v in (src_c, dst_f, src_f, dst_c):
            v.close()
    print(f"{case.name}: transfer worst {worst:.2e}")


def test_scale_eigenvalue_estimate(case):
    errs = {l: abs(case.gpu_lambda[l] / case.replica_lambda[l] - 1.0) for l in case.gpu_lambda}
    print(f"{case.name}: lambda {case.gpu_lambda}, relative deviation from the replica {errs}")
    assert max(errs.values()) <= TOL_LAMBDA, errs


def test_scale_smoother(case):
    mg, ref = case.mg, case.ref
    rng = np.random.default_rng(12)
    worst = 0.0
    for l in sorted({mg.n_levels - 1, (mg.n_levels - 1) // 2 + 1}):
        lop = mg.level_operator(l)
        b, x0 = _interior(rng, ref.bmask[l]), _interior(rng, ref.bmask[l])
        bv, xv = _vec(lop, b), _vec(lop)
        mg.smooth(l, xv, bv)
        e0 = _rel(xv.to_host(), ref.smooth(l, None, b))
        xv.import_host(x0)
        mg.smooth(l, xv, bv)
        e1 = _rel(xv.to_host(), ref.smooth(l, x0, b))
        bv.close(); xv.close()
        worst = max(worst, e0, e1)
        assert e0 <= TOL_SMOOTH and e1 <= TOL_SMOOTH, (case.name, l, e0, e1)
    print(f"{case.name}: smoother worst {worst:.2e}")


def test_scale_vcycle(case):
    mg, ref = case.mg, case.ref
    b = _interior(np.random.default_rng(13), ref.bmask[-1])
    bv, xv = _vec(case.op, b), _vec(case.op)
    mg.vmult(xv, bv)
    err = _rel(xv.to_host(), ref.vcycle(b))
    bv.close(); xv.close()
    print(f"{case.name}: V-cycle {err:.2e}")
    assert err <= TOL_VCYCLE, (case.name, err)


def test_scale_cg_from_nonzero_initial_guess(case):
    dc = _dc()
    op, mg, ref = case.op, case.mg, case.ref
    bv = _vec(op)
    op.assemble_rhs(bv)
    b = bv.to_host()
    x0 = _interior(np.random.default_rng(14), ref.bmask[-1])
    tol = 1e-10 * np.linalg.norm(b)
    xv = _vec(op, x0)
    ctl = dc.SolverControl(100, tol)
    dc.SolverCG(ctl).solve(op, xv, bv, preconditioner=mg)
    x_ref, its_ref, hist_ref = ref.solve(b, tol, x0=x0)
    hist_ref = np.array(hist_ref)
    # equal counts, unless the reference's last residual is so close to tol that round-off may decide
    if its_ref >= 1 and abs(hist_ref[-1] - tol) > 0.01 * tol:
        assert ctl.last_step() == its_ref, (case.name, ctl.last_step(), its_ref)
    n = min(ctl.last_step(), its_ref) + 1
    eh = float(np.max(np.abs(ctl.history[:n] - hist_ref[:n]) / hist_ref[:n]))
    ex = _rel(xv.to_host(), x_ref)
    print(f"{case.name}: MG-CG from x0 {ctl.last_step()} iterations (reference {its_ref}), history {eh:.2e}, "
          f"x {ex:.2e}")
    assert eh <= TOL_HIST and ex <= TOL_X, (case.name, eh, ex)
    # IterationNumberControl: success after exactly 2 steps from the same x0
    xv.import_host(x0)
    ctl = dc.IterationNumberControl(2, 1e-30)
    dc.SolverCG(ctl).solve(op, xv, bv, preconditioner=mg)
    assert ctl.last_step() == 2
    assert np.max(np.abs(ctl.history - hist_ref[:3]) / hist_ref[:3]) <= TOL_HIST
    bv.close(); xv.close()


# ---------------------------------------------------------------- parameter sweep on small hierarchies
SWEEP = {"p2": (2, (8, 4, 4), "gll", False), "p4": (4, (4, 4, 2), "gauss", True)}


def _small(gpu_ctx, key, **params):
    dc = _dc()
    p, cells, quad, helm = SWEEP[key]
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=QUADS[quad], operator_kind=int(helm),
                                                     deformation=1, eps=EPS))
    mg = dc.Multigrid(op, coarse_tol=1e-14, **params)
    ref = MatfreeMG(p, cells, quad=quad, helmholtz=helm, deform=1, eps=EPS,
                    degree=params.get("smoothing_degree", 5), smoothing_range=params.get("smoothing_range", 15.0),
                    eig_iterations=params.get("eig_iterations", 12))
    assert mg.n_levels == ref.n_levels >= 2 and np.any(~ref.bmask[0])
    return op, mg, ref


def _smooth_err(mg, ref, l, rng):
    lop = mg.level_operator(l)
    ref.lam[l] = mg.lambda_max(l)
    b, x0 = _interior(rng, ref.bmask[l]), _interior(rng, ref.bmask[l])
    bv, xv = _vec(lop, b), _vec(lop)
    mg.smooth(l, xv, bv)
    e0 = _rel(xv.to_host(), ref.smooth(l, None, b))
    xv.import_host(x0)
    mg.smooth(l, xv, bv)
    e1 = _rel(xv.to_host(), ref.smooth(l, x0, b))
    bv.close(); xv.close()
    return max(e0, e1)


@pytest.mark.parametrize("key", sorted(SWEEP))
@pytest.mark.parametrize("degree", [1, 2, 3, 8])
def test_smoothing_degree(gpu_ctx, key, degree):
    op, mg, ref = _small(gpu_ctx, key, smoothing_degree=degree)
    rng = np.random.default_rng(degree)
    for l in range(1, mg.n_levels):
        err = _smooth_err(mg, ref, l, rng)
        print(f"{key} smoothing_degree={degree} level {l}: smoother {err:.2e}")
        assert err <= TOL_SMOOTH, (key, degree, l, err)
    b = _interior(rng, ref.bmask[-1])
    bv, xv = _vec(op, b), _vec(op)
    mg.vmult(xv, bv)
    err = _rel(xv.to_host(), ref.vcycle(b))
    bv.close(); xv.close(); mg.close(); op.close()
    print(f"{key} smoothing_degree={degree}: V-cycle {err:.2e}")
    assert err <= TOL_VCYCLE, (key, degree, err)


@pytest.mark.parametrize("key", sorted(SWEEP))
@pytest.mark.parametrize("smoothing_range", [4.0, 30.0])
def test_smoothing_range(gpu_ctx, key, smoothing_range):
    op, mg, ref = _small(gpu_ctx, key, smoothing_range=smoothing_range)
    rng = np.random.default_rng(int(smoothing_range))
    for l in range(1, mg.n_levels):
        err = _smooth_err(mg, ref, l, rng)
        print(f"{key} smoothing_range={smoothing_range} level {l}: smoother {err:.2e}")
        assert err <= TOL_SMOOTH, (key, smoothing_range, l, err)
    mg.close(); op.close()


@pytest.mark.parametrize("key", sorted(SWEEP))
@pytest.mark.parametrize("eig_iterations", [1, 4, 20])
def test_eig_iterations(gpu_ctx, key, eig_iterations):
    op, mg, ref = _small(gpu_ctx, key, eig_iterations=eig_iterations)
    for l in range(1, mg.n_levels):
        got, want = mg.lambda_max(l), ref.estimate_lambda(l)
        print(f"{key} eig_iterations={eig_iterations} level {l}: lambda {got:.15g}, replica {want:.15g}")
        assert abs(got / want - 1.0) <= TOL_LAMBDA, (key, eig_iterations, l, got, want)
    mg.close(); op.close()


# ---------------------------------------------------------------- diagonal for every degree
# small deformed, anisotropic meshes whose cell count is not a multiple of cells_per_tile (32, 14, 8, 5, 3, 3, 2, 1
# for p = 1..8): the last tile has padded slots
DIAG_MESH = {1: (7, 5, 3), 2: (5, 4, 3), 3: (5, 3, 3), 4: (4, 3, 3), 5: (5, 2, 2), 6: (4, 2, 2), 7: (3, 3, 1),
             8: (3, 2, 2)}


@pytest.mark.parametrize("helmholtz", [False, True], ids=["poisson", "helm"])
@pytest.mark.parametrize("quad", ["gauss", "gll"])
@pytest.mark.parametrize("p", range(1, 9))
def test_diagonal_every_degree(gpu_ctx, p, quad, helmholtz):
    import re
    dc = _dc()
    cells = DIAG_MESH[p]
    upper = (1.5 * cells[0], 1.0 * cells[1], 0.75 * cells[2])
    op = dc.PoissonOperator(gpu_ctx, dc.make_problem(p, cells, quadrature=QUADS[quad], operator_kind=int(helmholtz),
                                                     upper=upper, deformation=1, eps=EPS))
    cpt = int(re.search(r"cells_per_tile=(\d+)", op.kernel_name).group(1))
    assert cpt == 1 or op.n_cells % cpt != 0, (op.kernel_name, op.n_cells)
    m = O.OracleMesh(p, cells, quad=QUADS[quad], upper=upper, deform=1, eps=EPS)
    d = _vec(op)
    op.compute_diagonal(d)
    got = _host(d)
    op.close()
    want = probe_diagonal(m, O.HELMHOLTZ if helmholtz else O.POISSON)
    print(f"diagonal p={p} {quad} {'Helmholtz' if helmholtz else 'Poisson'}: {_relmax(got, want):.2e}")
    assert _relmax(got, want) <= 1e-12, (p, quad, helmholtz, _relmax(got, want))
    assert _relmax(metric_diagonal(m, helmholtz), want) <= 1e-13
