"""Numpy/scipy restatement of the geometric multigrid preconditioner (csrc/mg.cu).

TEST INFRASTRUCTURE ONLY.  Level matrices come from NumpyBP5.assemble (assembled sparse, Dirichlet rows identity);
the prolongation is built along a different route from the library's: the position of every fine lattice node in
coarse-cell units, the 1D Lagrange basis of the coarse cell containing it evaluated there (product form), and
the Kronecker product P = P_z (x) P_y (x) P_x of the dense 1D matrices.  The smoother, V-cycle and outer CG follow
the algorithm of csrc/mg.cu step for step so that vectors can be compared.
"""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from bp5_numpy import NumpyBP5, lobatto01


def lagrange_values(nodes, x):
    """phi_a(x) of the Lagrange basis through `nodes`, product form (the monomial route of lagrange_tables loses
    about three digits at p = 8, too many for a 1e-13 check)"""
    n = len(nodes)
    out = np.ones(n)
    for a in range(n):
        for b in range(n):
            if b != a:
                out[a] *= (x - nodes[b]) / (nodes[a] - nodes[b])
    return out


def prolongation_1d(p, c):
    """(2 p c + 1) x (p c + 1): nodal interpolation from c coarse cells to 2c fine cells of degree p"""
    xi, _ = lobatto01(p + 1)
    nf, nc = 2 * p * c + 1, p * c + 1
    P = np.zeros((nf, nc))
    for f in range(nf):
        fc = min(f // p, 2 * c - 1)
        pos = 0.5 * (fc + xi[f - fc * p])          # in coarse-cell units
        cc = min(int(np.floor(pos)), c - 1)
        P[f, cc * p: cc * p + p + 1] = lagrange_values(xi, pos - cc)
    return P


def prolongation(p, coarse_cells):
    """P = P_z (x) P_y (x) P_x on the lexicographic lattice (x fastest)"""
    Px, Py, Pz = (sp.csr_matrix(prolongation_1d(p, c)) for c in coarse_cells)
    return sp.kron(Pz, sp.kron(Py, Px)).tocsr()


def level_cells(cells, max_levels=0):
    """cell counts of the levels, coarsest first: halve while every count is even"""
    out = [tuple(cells)]
    while (max_levels == 0 or len(out) < max_levels) and all(c % 2 == 0 for c in out[-1]):
        out.append(tuple(c // 2 for c in out[-1]))
    return out[::-1]


class NumpyMG:
    """Levels, transfer, Chebyshev-Jacobi smoother, V-cycle and preconditioned CG.
    lambdas: {level: estimate of lambda_max(D^-1 A)} (default: the exact value from eigsh on the interior);
    coarse_tol None: exact coarse solve (splu on the interior rows), else Jacobi CG to coarse_tol |b|."""

    def __init__(self, p, cells, quad="gauss", helmholtz=False, deform=0, eps=0.0, upper=None, max_levels=0,
                 degree=5, smoothing_range=15.0, coarse_tol=None, coarse_max_its=1000, lambdas=None):
        upper = tuple(float(c) for c in cells) if upper is None else tuple(upper)
        self.p, self.degree, self.range = p, degree, smoothing_range
        self.coarse_tol, self.coarse_max_its = coarse_tol, coarse_max_its
        self.cells = level_cells(cells, max_levels)
        self.n_levels = len(self.cells)
        self.meshes, self.A, self.dinv, self.bmask, self.P = [], [], [], [], [None]
        for l, c in enumerate(self.cells):
            m = NumpyBP5(p, c, quad=quad, upper=upper, deform=deform, eps=eps)   # same domain on every level
            A = m.assemble(helmholtz=helmholtz)
            self.meshes.append(m)
            self.A.append(A)
            self.dinv.append(1.0 / A.diagonal())
            self.bmask.append(m.boundary_mask())
            if l > 0:
                self.P.append(prolongation(p, self.cells[l - 1]))
        self.lam = {}
        for l in range(1, self.n_levels):
            self.lam[l] = lambdas[l] if lambdas and l in lambdas else self.exact_lambda(l)
        inner = ~self.bmask[0]
        self._coarse_lu = spla.splu(self.A[0][inner][:, inner].tocsc()) if coarse_tol is None else None

    def exact_lambda(self, l):
        inner = ~self.bmask[l]
        Ai = self.A[l][inner][:, inner]
        s = sp.diags(np.sqrt(self.dinv[l][inner]))
        return float(spla.eigsh((s @ Ai @ s).tocsc(), k=1, which="LA", return_eigenvectors=False)[0])

    def prolongate(self, l, xc):
        return self.P[l] @ xc

    def restrict(self, l, rf):
        out = self.P[l].T @ rf
        out[self.bmask[l - 1]] = 0.0
        return out

    def smooth(self, l, x, b):
        """Chebyshev smoothing from x (None: zero), as csrc/mg.cu"""
        A, Di = self.A[l], self.dinv[l]
        lmax = 1.2 * self.lam[l]
        lmin = lmax / self.range
        theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
        sigma = theta / delta
        rho0 = 1.0 / sigma
        if x is None:
            x = np.zeros_like(b)
            r = b.copy()
        else:
            x = x.copy()
            r = b - A @ x
        d = Di * r / theta
        for j in range(1, self.degree + 1):
            x += d
            if j == self.degree:
                break
            r -= A @ d
            rho1 = 1.0 / (2.0 * sigma - rho0)
            d = rho1 * rho0 * d + (2.0 * rho1 / delta) * Di * r
            rho0 = rho1
        return x

    def coarse(self, b):
        if self._coarse_lu is not None:
            inner = ~self.bmask[0]
            x = b.copy()
            x[inner] = self._coarse_lu.solve(b[inner])
            return x
        x, _, _ = pcg(lambda v: self.A[0] @ v, lambda g: self.dinv[0] * g, b,
                      self.coarse_tol * np.linalg.norm(b), self.coarse_max_its)
        return x

    def vcycle(self, b, l=None):
        l = self.n_levels - 1 if l is None else l
        if l == 0:
            return self.coarse(b)
        x = self.smooth(l, None, b)
        r = b - self.A[l] @ x
        xc = self.vcycle(self.restrict(l, r), l - 1)
        x = x + self.prolongate(l, xc)
        return self.smooth(l, x, b)

    def solve(self, b, tol, max_its=100):
        """MG-preconditioned standard CG from x = 0: (x, iterations, residual history)"""
        return pcg(lambda v: self.A[-1] @ v, self.vcycle, b, tol, max_its)


def dot(a, b):
    """a . b through numpy's own loops: a BLAS level-1 call leaves OpenBLAS's worker threads spinning, and they slow
    the next OpenMP oracle vmult (mg_matfree.py) by an order of magnitude"""
    return float(np.einsum("i,i->", a, b))


def pcg(apply_A, apply_M, b, tol, max_its, x0=None):
    """dealii::SolverCG with a preconditioner from x0 (None: zero; stops at |g| <= tol or max_its)"""
    if x0 is None:
        x = np.zeros_like(b)
        g = -b.copy()
    else:
        x = np.array(x0, dtype=np.float64)
        g = apply_A(x) - b
    res = np.sqrt(dot(g, g))
    hist = [res]
    if res <= tol or max_its == 0:
        return x, 0, hist
    h = apply_M(g)
    d = -h
    gh = dot(g, h)
    it = 0
    while True:
        it += 1
        ad = apply_A(d)
        alpha = gh / dot(d, ad)
        x += alpha * d
        g += alpha * ad
        res = np.sqrt(dot(g, g))
        hist.append(res)
        if res <= tol or it >= max_its:
            break
        h = apply_M(g)
        gh_old, gh = gh, dot(g, h)
        d = (gh / gh_old) * d - h
    return x, it, hist
