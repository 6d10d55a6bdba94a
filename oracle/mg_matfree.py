"""Matrix-free restatement of the geometric multigrid preconditioner (csrc/mg.cu) that scales to millions of DoFs.

TEST INFRASTRUCTURE ONLY.  oracle/mg_numpy.py assembles every level as a sparse matrix and so stops at a few thousand
DoFs; this module applies every level operator with the C++ oracle's OpenMP, matrix-free OracleMesh.vmult (semantics
0, what level_vmult does: the cell loop over the unconstrained operator, then dst = src on the Dirichlet rows).

  * levels: one OracleMesh per level, cells halved while all counts are even (mg_numpy.level_cells); every level
    has the finest mesh's domain, deformation and quadrature, as bp5_mg_create builds them.
  * transfer: P = P_z (x) P_y (x) P_x applied as three dense 1D contractions on the (z, y, x) lattice with
    mg_numpy.prolongation_1d (nodal interpolation, product-form Lagrange basis); R = P^T the same way, coarse
    Dirichlet rows zeroed.  No sparse Kronecker product is formed.
  * inverse diagonal, independent of diagonal_kernel: the separable element-diagonal formula on the oracle's merged
    metric (planes xx, yy, zz, xy, xz, yz, JxW included) with per-direction factors Dg Dg, B Dg and B B, plus for
    Helmholtz the mass term a(x_q) JxW B B B; summed over the cells sharing a DoF, Dirichlet rows 1.
    probe_diagonal() reads the same diagonal off (p+1)^3 oracle vmults (one per residue class of the lattice index
    mod p+1 in each direction: DoFs of one class never share a cell) and serves as the cross-check.
  * Chebyshev smoother, V-cycle and preconditioned CG exactly as mg_numpy.NumpyMG; the CG takes an initial guess.
    The coarsest level is solved to round-off by Jacobi-preconditioned CG on the oracle operator.
  * estimate_lambda: a replica of csrc/mg.cu's estimate, start vector included -- mg_random_fill (splitmix64 of
    i + 1, seed 0x5eed + level) in numpy uint64 arithmetic, zeroed on the Dirichlet rows -- then `eig_iterations`
    Jacobi-PCG steps with the C++ loop's break conditions, the same Lanczos tridiagonal T and its largest
    eigenvalue.  It reproduces the library's estimate, not the exact lambda_max: if the start vector or the
    iteration in csrc/mg.cu is changed on purpose, this replica has to change with it.
"""
import numpy as np

import oracle as O
from mg_numpy import dot, level_cells, pcg, prolongation_1d


def random_fill(n, seed):
    """mg_random_fill: uniform in [-1, 1) from the splitmix64 hash of i + 1"""
    z = np.uint64(seed) + np.uint64(0x9e3779b97f4a7c15) * (np.arange(n, dtype=np.uint64) + np.uint64(1))
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xbf58476d1ce4e5b9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94d049bb133111eb)
    z ^= z >> np.uint64(31)
    return (z >> np.uint64(11)).astype(np.float64) * (2.0 / 9007199254740992.0) - 1.0


def lanczos_lambda_max(alpha, beta):
    """largest eigenvalue of the Lanczos tridiagonal of the CG coefficients, built as in estimate_lambda"""
    m = len(alpha)
    T = np.zeros((m, m))
    for j in range(m):
        T[j, j] = 1.0 / alpha[j] + (beta[j - 1] / alpha[j - 1] if j > 0 else 0.0)
        if j + 1 < m:
            T[j, j + 1] = T[j + 1, j] = np.sqrt(beta[j]) / alpha[j]
    return float(np.linalg.eigvalsh(T)[-1])


def _contract3(planes, fx, fy, fz):
    """sum_q plane[c, q] fx[qx, i] fy[qy, j] fz[qz, k] -> [c, (k, j, i)] (q and the result x fastest)"""
    n = fx.shape[0]
    v = planes.reshape(-1, n, n, n)                      # [c, qz, qy, qx]
    v = v @ fx                                           # [c, qz, qy, i]
    v = np.einsum("czyi,yj->czji", v, fy)
    v = np.einsum("czji,zk->ckji", v, fz)
    return v.reshape(-1, n ** 3)


def metric_diagonal(mesh, helmholtz=False):
    """diagonal of the level operator from the oracle's metric (Dirichlet rows 1)"""
    sh = O.shape(mesh.p, mesh.quad)
    B, Dg = sh["B"], sh["Dg"]
    BB, DD, BD = B * B, Dg * Dg, B * Dg
    G = mesh.metric()
    cell = _contract3(G[0], DD, BB, BB)
    cell += _contract3(G[1], BB, DD, BB)
    cell += _contract3(G[2], BB, BB, DD)
    cell += 2.0 * _contract3(G[3], BD, BD, BB)
    cell += 2.0 * _contract3(G[4], BD, BB, BD)
    cell += 2.0 * _contract3(G[5], BB, BD, BD)
    del G
    l2g = O._cell_dofs(mesh)
    if helmholtz:   # + sum_q a(x_q) JxW phi_i(q)^2, a = 10 / (0.05 + 2 |x_q|^2) (step-64's coefficient)
        X = mesh.dof_coords()
        xq2 = sum(O._interp3(B, X[:, d][l2g]) ** 2 for d in range(3))
        cell += _contract3(10.0 / (0.05 + 2.0 * xq2) * mesh.jxw(), BB, BB, BB)
    diag = np.bincount(l2g.ravel(), weights=cell.ravel(), minlength=mesh.n_dofs)
    diag[mesh.boundary_mask()] = 1.0
    return diag


def probe_diagonal(mesh, kind):
    """diagonal of the level operator read off (p+1)^3 oracle vmults, one per residue class of the lattice index"""
    n = mesh.p + 1
    idx = [np.arange(nd) % n for nd in mesh.nd]            # x, y, z
    diag = np.zeros(mesh.n_dofs)
    for rz in range(n):
        for ry in range(n):
            for rx in range(n):
                sel = ((idx[2] == rz)[:, None, None] & (idx[1] == ry)[None, :, None]
                       & (idx[0] == rx)[None, None, :]).ravel()
                out = mesh.vmult(sel.astype(np.float64), kind=kind, semantics=0)
                diag[sel] = out[sel]
    return diag


class MatfreeMG:
    """Levels, transfer, smoother, V-cycle, MG-preconditioned CG and the eigenvalue estimate replica.
    lambdas: {level: lambda_max used by the smoother}; a level without one uses estimate_lambda(level)."""

    def __init__(self, p, cells, quad="gauss", helmholtz=False, deform=0, eps=0.0, max_levels=0, degree=5,
                 smoothing_range=15.0, eig_iterations=12, lambdas=None, coarse_rtol=1e-15, coarse_max_its=20000):
        self.p, self.degree, self.range, self.eig_its = p, degree, smoothing_range, eig_iterations
        self.kind = O.HELMHOLTZ if helmholtz else O.POISSON
        self.coarse_rtol, self.coarse_max_its = coarse_rtol, coarse_max_its
        self.cells = level_cells(cells, max_levels)
        self.n_levels = len(self.cells)
        upper = tuple(float(c) for c in cells)              # make_problem's default: unit cells on the finest level
        qk = O.GLL if quad == "gll" else O.GAUSS
        self.meshes = [O.OracleMesh(p, c, quad=qk, upper=upper, deform=deform, eps=eps) for c in self.cells]
        self.bmask = [m.boundary_mask() for m in self.meshes]
        self.dinv = [1.0 / metric_diagonal(m, helmholtz) for m in self.meshes]
        self.P1 = [None] + [[prolongation_1d(p, c) for c in self.cells[l - 1]] for l in range(1, self.n_levels)]
        self.lam = dict(lambdas or {})
        self.coarse_its = []                                # iterations of every coarse solve (diagnostics)

    def n(self, l):
        return self.meshes[l].n_dofs

    def vmult(self, l, src):
        return self.meshes[l].vmult(src, kind=self.kind, semantics=0)

    # ---- transfer
    def prolongate(self, l, xc):
        Px, Py, Pz = self.P1[l]
        nx, ny, nz = self.meshes[l - 1].nd
        v = xc.reshape(nz, ny, nx) @ Px.T                   # [nz, ny, NX]
        v = np.matmul(Py, v)                                # [nz, NY, NX]
        return (Pz @ v.reshape(nz, -1)).ravel()

    def restrict(self, l, rf):
        Px, Py, Pz = self.P1[l]
        NX, NY, NZ = self.meshes[l].nd
        v = (Pz.T @ rf.reshape(NZ, -1)).reshape(-1, NY, NX)   # [nz, NY, NX]
        v = np.matmul(Py.T, v)                                # [nz, ny, NX]
        out = (v @ Px).ravel()
        out[self.bmask[l - 1]] = 0.0
        return out

    # ---- smoother, coarse solve, V-cycle, CG
    def lambda_max(self, l):
        if l not in self.lam:
            self.lam[l] = self.estimate_lambda(l)
        return self.lam[l]

    def smooth(self, l, x, b):
        """Chebyshev smoothing from x (None: zero), as csrc/mg.cu and mg_numpy.NumpyMG.smooth"""
        Di = self.dinv[l]
        lmax = 1.2 * self.lambda_max(l)
        lmin = lmax / self.range
        theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
        sigma = theta / delta
        rho0 = 1.0 / sigma
        if x is None:
            x = np.zeros_like(b)
            r = b.copy()
        else:
            x = x.copy()
            r = b - self.vmult(l, x)
        d = Di * r / theta
        for j in range(1, self.degree + 1):
            x += d
            if j == self.degree:
                break
            r -= self.vmult(l, d)
            rho1 = 1.0 / (2.0 * sigma - rho0)
            d = rho1 * rho0 * d + (2.0 * rho1 / delta) * Di * r
            rho0 = rho1
        return x

    def coarse(self, b):
        """level 0 solved to round-off: Jacobi-PCG until the residual is coarse_rtol |b|"""
        x, its, _ = pcg(lambda v: self.vmult(0, v), lambda g: self.dinv[0] * g, b,
                        self.coarse_rtol * np.sqrt(dot(b, b)), self.coarse_max_its)
        self.coarse_its.append(its)
        return x

    def vcycle(self, b, l=None):
        l = self.n_levels - 1 if l is None else l
        if l == 0:
            return self.coarse(b)
        x = self.smooth(l, None, b)
        r = b - self.vmult(l, x)
        xc = self.vcycle(self.restrict(l, r), l - 1)
        return self.smooth(l, x + self.prolongate(l, xc), b)

    def solve(self, b, tol, max_its=100, x0=None):
        """MG-preconditioned standard CG: (x, iterations, residual history)"""
        return pcg(lambda v: self.vmult(self.n_levels - 1, v), self.vcycle, b, tol, max_its, x0=x0)

    # ---- eigenvalue estimate
    def estimate_lambda(self, l):
        """replica of estimate_lambda (csrc/mg.cu) on level l >= 1"""
        Di = self.dinv[l]
        r = random_fill(self.n(l), 0x5eed + l)
        r[self.bmask[l]] = 0.0
        z = Di * r
        p = z.copy()
        rz = dot(r, z)
        alpha, beta = [], []
        j = 0
        while j < self.eig_its and rz > 0.0:
            q = self.vmult(l, p)
            pq = dot(p, q)
            if not pq > 0.0:
                break
            a = rz / pq
            alpha.append(a)
            r -= a * q
            z = Di * r
            rz_new = dot(r, z)
            bt = rz_new / rz
            rz = rz_new
            if j + 1 < self.eig_its and rz > 0.0:
                beta.append(bt)
                p = bt * p + z
            j += 1
        assert alpha, "eigenvalue estimate: no CG step possible"
        return lanczos_lambda_max(alpha, beta)
