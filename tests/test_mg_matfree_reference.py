"""CPU checks of the matrix-free multigrid reference (oracle/mg_matfree.py) against the assembled one
(oracle/mg_numpy.py) on small meshes.  The GPU multigrid is compared with the matrix-free reference at millions of
DoFs (tests/test_gpu_multigrid_scale.py), so a wrong reference is the first thing to rule out: transfer, diagonal,
smoother, V-cycle and preconditioned CG from a non-zero initial guess must agree with the assembled reference to
round-off, the metric and probed diagonals with each other, and the eigenvalue estimate replica with the exact
largest eigenvalue once the Lanczos process has run to convergence."""
import functools

import numpy as np
import pytest

from mg_matfree import MatfreeMG, lanczos_lambda_max, metric_diagonal, probe_diagonal, random_fill
from mg_numpy import NumpyMG

# (p, cells, quad, helmholtz, deform): three levels each, and the coarsest level has interior DoFs
CASES = [(2, (8, 4, 4), "gauss", False, 0), (3, (8, 4, 4), "gll", True, 1)]
IDS = ["p2-gauss-poisson", "p3-gll-helmholtz-deformed"]


@functools.lru_cache(maxsize=None)
def _pair(p, cells, quad, helmholtz, deform):
    """(matrix-free, assembled) references on the same levels; the assembled one solves the coarsest level with LU
    and both use the matrix-free replica's eigenvalue estimates"""
    mf = MatfreeMG(p, cells, quad=quad, helmholtz=helmholtz, deform=deform, eps=0.1 if deform else 0.0)
    lam = {l: mf.lambda_max(l) for l in range(1, mf.n_levels)}
    ref = NumpyMG(p, cells, quad=quad, helmholtz=helmholtz, deform=deform, eps=0.1 if deform else 0.0, lambdas=lam)
    assert mf.cells == ref.cells and mf.n_levels == 3
    assert np.any(~mf.bmask[0])
    return mf, ref


def _interior(rng, mask):
    u = rng.standard_normal(mask.size)
    u[mask] = 0.0
    return u


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _relmax(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_transfer_matches_kronecker_prolongation(case):
    mf, ref = _pair(*case)
    rng = np.random.default_rng(1)
    for l in range(1, mf.n_levels):
        uc, uf = rng.standard_normal(mf.n(l - 1)), rng.standard_normal(mf.n(l))
        assert _relmax(mf.prolongate(l, uc), ref.prolongate(l, uc)) <= 1e-14, l
        assert _relmax(mf.restrict(l, uf), ref.restrict(l, uf)) <= 1e-14, l


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_diagonal_matches_assembled_and_probed(case):
    mf, ref = _pair(*case)
    for l in range(mf.n_levels):
        d_metric, d_asm = 1.0 / mf.dinv[l], 1.0 / ref.dinv[l]
        d_probe = probe_diagonal(mf.meshes[l], mf.kind)
        assert _relmax(d_metric, d_asm) <= 1e-13, l
        assert _relmax(d_probe, d_asm) <= 1e-13, l
        assert _relmax(d_metric, d_probe) <= 1e-13, l


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_smoother_and_vcycle_match_assembled(case):
    mf, ref = _pair(*case)
    rng = np.random.default_rng(2)
    for l in range(1, mf.n_levels):
        b, x0 = _interior(rng, mf.bmask[l]), _interior(rng, mf.bmask[l])
        assert _rel(mf.smooth(l, None, b), ref.smooth(l, None, b)) <= 1e-12, l
        assert _rel(mf.smooth(l, x0, b), ref.smooth(l, x0, b)) <= 1e-12, l
    b = _interior(rng, mf.bmask[-1])
    assert _rel(mf.vcycle(b), ref.vcycle(b)) <= 1e-12


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_pcg_from_nonzero_guess_matches_assembled(case):
    from mg_numpy import pcg
    mf, ref = _pair(*case)
    rng = np.random.default_rng(3)
    b = ref.meshes[-1].rhs()
    x0 = _interior(rng, mf.bmask[-1])
    tol = 1e-10 * np.linalg.norm(b)
    x, its, hist = mf.solve(b, tol, x0=x0)
    xr, its_r, hist_r = pcg(lambda v: ref.A[-1] @ v, ref.vcycle, b, tol, 100, x0=x0)
    assert its == its_r and 3 <= its <= 20, (its, its_r)
    assert np.max(np.abs(np.array(hist) - hist_r) / np.array(hist_r)) <= 1e-11
    assert hist[0] == pytest.approx(np.linalg.norm(ref.A[-1] @ x0 - b), rel=1e-13)   # g = A x0 - b, not -b
    assert _rel(x, xr) <= 1e-11


def test_helmholtz_metric_diagonal_matches_probing_on_an_anisotropic_mesh():
    import oracle as O
    for p in (1, 5):
        m = O.OracleMesh(p, (3, 2, 5), quad=O.GAUSS, upper=(1.0, 3.0, 2.0), deform=1, eps=0.1)
        assert _relmax(metric_diagonal(m, helmholtz=True), probe_diagonal(m, O.HELMHOLTZ)) <= 1e-13, p


def test_random_fill_is_splitmix64():
    """the numpy uint64 replica against Python's arbitrary-precision integers"""
    def one(i, seed):
        M = (1 << 64) - 1
        z = (seed + 0x9e3779b97f4a7c15 * (i + 1)) & M
        z = ((z ^ (z >> 30)) * 0xbf58476d1ce4e5b9) & M
        z = ((z ^ (z >> 27)) * 0x94d049bb133111eb) & M
        z ^= z >> 31
        return (z >> 11) * (2.0 / 9007199254740992.0) - 1.0
    seed = 0x5eed + 3
    v = random_fill(1000, seed)
    assert all(v[i] == one(i, seed) for i in (0, 1, 2, 499, 999))
    assert -1.0 <= v.min() and v.max() < 1.0 and abs(v.mean()) < 0.1


def test_eigenvalue_replica_converges_to_the_exact_value():
    """run to convergence, the Lanczos tridiagonal's largest eigenvalue is lambda_max(D^-1 A): a wrong entry of T
    would leave it off; at the default 12 steps the estimate sits a little below"""
    mf, ref = _pair(*CASES[0])
    for l in range(1, mf.n_levels):
        exact = ref.exact_lambda(l)
        assert 0.9 * exact <= mf.lambda_max(l) <= (1.0 + 1e-12) * exact
        mf_long = MatfreeMG(2, mf.cells[l], eig_iterations=60)
        assert mf_long.estimate_lambda(mf_long.n_levels - 1) == pytest.approx(exact, rel=1e-8), l
    # T of the CG coefficients of a diagonal matrix: the eigenvalues are the matrix's
    lam = np.array([1.0, 2.0, 5.0])
    r = np.ones(3)
    p, rz, alpha, beta = r.copy(), r @ r, [], []
    for j in range(3):
        q = lam * p
        a = rz / (p @ q)
        alpha.append(a)
        r = r - a * q
        rz_new = r @ r
        if j + 1 < 3:
            beta.append(rz_new / rz)
            p = r + beta[-1] * p
        rz = rz_new
    assert lanczos_lambda_max(alpha, beta) == pytest.approx(5.0, rel=1e-12)
