"""numpy/scipy restatement of the multigrid path of ``fea_batch_set_refinement`` (TEST INFRASTRUCTURE).

Mirrors ``fea_diffusion_b200/csrc/k_mg.cu`` (DESIGN.md section 3.9): the hierarchy of a uniform red
refinement (``workload.refine_uniform`` numbering), the prolongation P, the Galerkin coarse operators
summed cell by cell, and flexible CG preconditioned by a Chebyshev-smoothed V-cycle in the
2x2-block-Jacobi-scaled spaces.  The coarsest level is solved exactly (sparse LU) here.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from .fea_oracle import assemble_csr, element_stiffness, equation_map, fix_orientation


def hierarchy(conn: np.ndarray, levels: int) -> Tuple[List[np.ndarray], List[Optional[np.ndarray]]]:
    """(conns, parents), coarsest level first.  conns[l] is level l's connectivity in the numbering as
    given; parents[l] (l >= 1) is (n_v(l), 2): (v, -1) for a vertex of level l-1, else the ends of the
    level-(l-1) edge whose midpoint it is.  Children of coarse cell p are p, p+nc, p+2nc, p+3nc =
    (a,ab,ca), (ab,b,bc), (ca,bc,c), (ab,bc,ca)."""
    conns = [np.asarray(conn, dtype=np.int64)]
    pars: List[Optional[np.ndarray]] = []
    for _ in range(levels):
        cf = conns[0]
        nc = len(cf) // 4
        c0, c1, c2 = cf[:nc], cf[nc:2 * nc], cf[2 * nc:3 * nc]
        a, b, c = c0[:, 0], c1[:, 1], c2[:, 2]
        cc = np.stack([a, b, c], 1)
        nvc, nvf = int(cc.max()) + 1, int(cf.max()) + 1
        par = np.full((nvf, 2), -1, dtype=np.int64)
        par[:nvc, 0] = np.arange(nvc)
        for m, u, w in ((c0[:, 1], a, b), (c1[:, 2], b, c), (c0[:, 2], c, a)):
            par[m, 0] = np.minimum(u, w)
            par[m, 1] = np.maximum(u, w)
        conns.insert(0, cc)
        pars.insert(0, par)
    return conns, [None] + pars


def prolongation(par: np.ndarray, n_coarse: int) -> sp.csr_matrix:
    """P over all DOFs (2 n_fine x 2 n_coarse): weight 1 from the same vertex, 1/2 from each edge end."""
    nvf = len(par)
    rows, cols, vals = [], [], []
    own = par[:, 1] < 0
    for comp in range(2):
        f = np.flatnonzero(own)
        rows.append(2 * f + comp), cols.append(2 * par[f, 0] + comp), vals.append(np.ones(len(f)))
        f = np.flatnonzero(~own)
        for e in range(2):
            rows.append(2 * f + comp), cols.append(2 * par[f, e] + comp), vals.append(np.full(len(f), 0.5))
    return sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(2 * nvf, 2 * n_coarse))


def galerkin_cells(conn_f: np.ndarray, ke_f: np.ndarray, fixed_f: np.ndarray, par_f: np.ndarray,
                   conn_c: np.ndarray) -> np.ndarray:
    """6x6 matrix of every coarse cell: sum over its four children of P_e^T M K_e M P_e (conn_f / conn_c
    in the orientation the element matrices use; M zeroes the DOFs fixed on the fine level)."""
    nc = len(conn_c)
    kc = np.zeros((nc, 6, 6))
    fixed_f = np.asarray(fixed_f, dtype=bool)
    for k in range(4):
        F = conn_f[k * nc:(k + 1) * nc]
        pr = par_f[F]                                   # (nc, 3, 2)
        wx = np.where(pr[:, :, 1] < 0, 1.0, 0.5) * ~fixed_f[F]
        wy = np.where(pr[:, :, 1] < 0, 0.0, 0.5) * ~fixed_f[F]
        W = (wx[:, :, None] * (conn_c[:, None, :] == pr[:, :, 0:1]) +
             wy[:, :, None] * (conn_c[:, None, :] == pr[:, :, 1:2]))   # (nc, 3 fine, 3 coarse)
        Pe = np.einsum("naj,cd->nacjd", W, np.eye(2)).reshape(nc, 6, 6)
        kc += np.einsum("nai,nab,nbj->nij", Pe, ke_f[k * nc:(k + 1) * nc], Pe)
    return kc


def block_scaling(K: sp.csr_matrix) -> sp.csr_matrix:
    """S = blockdiag(L_v^-T) of the 2x2 diagonal blocks: S^T K S has identity diagonal blocks."""
    n = K.shape[0] // 2
    d = K.diagonal()
    dc = np.asarray(K[np.arange(0, 2 * n, 2), np.arange(1, 2 * n, 2)]).ravel()
    l00 = np.sqrt(d[0::2])
    l10 = dc / l00
    l11 = np.sqrt(d[1::2] - l10 * l10)
    i00, i11 = 1.0 / l00, 1.0 / l11
    i10 = -l10 * i00 * i11
    r = np.arange(n)
    rows = np.concatenate([2 * r, 2 * r, 2 * r + 1])
    cols = np.concatenate([2 * r, 2 * r + 1, 2 * r + 1])
    return sp.csr_matrix((np.concatenate([i00, i10, i11]), (rows, cols)), shape=(2 * n, 2 * n))


class Multigrid:
    """Hierarchy, operators and preconditioner of one uniformly refined problem (coors, conn as given,
    cell_region, D per region, fixed vertices); level 0 is the coarsest."""

    def __init__(self, coors, conn, cell_region, D, fixed, levels: int, degree: int = 3, lanczos_steps: int = 20):
        coors = np.asarray(coors, dtype=np.float64)
        fixed = np.asarray(fixed, dtype=bool)
        cell_region = np.asarray(cell_region)
        conns, self.parents = hierarchy(conn, levels)
        self.levels, self.degree = levels, degree
        nvs = [int(c.max()) + 1 for c in conns]
        nvs[-1] = len(coors)
        oriented = [fix_orientation(coors[:nv], c)[0] for nv, c in zip(nvs, conns)]
        creg = [cell_region[:len(c)] for c in conns]   # children p, p+nc, ... share the region of parent p
        Dc = np.asarray(D)[np.maximum(cell_region, 0)]
        ke = element_stiffness(coors, oriented[-1], Dc)
        ke[cell_region < 0] = 0.0
        self.ke = [None] * (levels + 1)
        self.ke[levels] = ke
        for l in range(levels, 0, -1):
            self.ke[l - 1] = galerkin_cells(oriented[l], self.ke[l], fixed[:nvs[l]], self.parents[l], oriented[l - 1])
        self.K = [assemble_csr(nvs[l], oriented[l], self.ke[l], creg[l], fixed[:nvs[l]]) for l in range(levels + 1)]
        self.n_vertices, self.conns, self.oriented, self.fixed = nvs, conns, oriented, fixed
        # reduced P between consecutive levels, then everything in the scaled spaces
        self.P = [None]
        for l in range(1, levels + 1):
            eq_f, _ = equation_map(fixed[:nvs[l]])
            eq_c, _ = equation_map(fixed[:nvs[l - 1]])
            self.P.append(prolongation(self.parents[l], nvs[l - 1])[eq_f >= 0][:, eq_c >= 0].tocsr())
        self.S = [block_scaling(K) for K in self.K]
        self.Kh = [(S.T @ K @ S).tocsr() for S, K in zip(self.S, self.K)]
        self.Ph = [None] + [(_block_inverse(self.S[l]) @ self.P[l] @ self.S[l - 1]).tocsr() for l in range(1, levels + 1)]
        self.lmax = [_lanczos_lmax(A, lanczos_steps) for A in self.Kh]
        self.coarse = spla.splu(self.Kh[0].tocsc())

    def galerkin_reference(self, l: int) -> sp.csr_matrix:
        """P^T K_(l+1) P by sparse products (what the cell-by-cell sum must equal)."""
        return (self.P[l + 1].T @ self.K[l + 1] @ self.P[l + 1]).tocsr()

    def _cheb(self, l, b, x):
        A = self.Kh[l]
        hi, lo = 1.1 * self.lmax[l], self.lmax[l] / 30.0
        theta, delta = 0.5 * (hi + lo), 0.5 * (hi - lo)
        sigma = theta / delta
        rho = 1.0 / sigma
        r = b - A @ x
        d = r / theta
        for k in range(self.degree):
            x = x + d
            if k == self.degree - 1:
                break
            r = r - A @ d
            rn = 1.0 / (2.0 * sigma - rho)
            d = rn * rho * d + (2.0 * rn / delta) * r
            rho = rn
        return x

    def vcycle(self, b: np.ndarray, l: Optional[int] = None) -> np.ndarray:
        """z = M b in the scaled space of level l (default: the finest)."""
        l = self.levels if l is None else l
        if l == 0:
            return self.coarse.solve(b)
        x = self._cheb(l, b, np.zeros_like(b))
        r = b - self.Kh[l] @ x
        x = x + self.Ph[l] @ self.vcycle(self.Ph[l].T @ r, l - 1)
        return self._cheb(l, b, x)

    def apply_unscaled(self, r: np.ndarray) -> np.ndarray:
        """z = S M S^T r on active DOFs of the finest level (fea_batch_mg_apply)."""
        S = self.S[self.levels]
        return S @ self.vcycle(S.T @ r)

    def solve(self, f: np.ndarray, rtol: float = 1e-10, max_iter: int = 200) -> Tuple[np.ndarray, int]:
        """Flexible CG on the finest level for K u = f (active DOFs): (u, outer iterations)."""
        S, A = self.S[self.levels], self.Kh[self.levels]
        b = S.T @ f
        x = np.zeros_like(b)
        r = b.copy()
        tol = rtol * np.linalg.norm(b)
        p = q = None
        rz_old = alpha = 0.0
        it = 0
        while np.linalg.norm(r) > tol and it < max_iter:
            z = self.vcycle(r)
            rz = r @ z
            # flexible CG: beta = z+.(r+ - r) / (r.z), and r+ - r = -alpha q
            p = z if p is None else z + (-alpha * (z @ q) / rz_old) * p
            q = A @ p
            alpha = rz / (p @ q)
            x += alpha * p
            r -= alpha * q
            rz_old = rz
            it += 1
        return S @ x, it


def _block_inverse(S: sp.csr_matrix) -> sp.csr_matrix:
    """Inverse of a 2x2-block-diagonal upper-triangular S."""
    n = S.shape[0] // 2
    r = np.arange(n)
    i00 = np.asarray(S[2 * r, 2 * r]).ravel()
    i10 = np.asarray(S[2 * r, 2 * r + 1]).ravel()
    i11 = np.asarray(S[2 * r + 1, 2 * r + 1]).ravel()
    rows = np.concatenate([2 * r, 2 * r, 2 * r + 1])
    cols = np.concatenate([2 * r, 2 * r + 1, 2 * r + 1])
    return sp.csr_matrix((np.concatenate([1.0 / i00, -i10 / (i00 * i11), 1.0 / i11]), (rows, cols)), shape=S.shape)


def _lanczos_lmax(A: sp.csr_matrix, steps: int) -> float:
    """Top Ritz value of ``steps`` Lanczos steps from a random vector (the device's lambda_max estimate)."""
    v = np.random.default_rng(0).uniform(-1.0, 1.0, A.shape[0])
    v /= np.linalg.norm(v)
    vp = np.zeros_like(v)
    alpha, beta = [], []
    b = 0.0
    for _ in range(steps):
        w = A @ v
        a = v @ w
        w = w - a * v - b * vp
        b = np.linalg.norm(w)
        alpha.append(a)
        beta.append(b)
        if b == 0.0:
            break
        vp, v = v, w / b
    T = np.diag(alpha) + np.diag(beta[:len(alpha) - 1], 1) + np.diag(beta[:len(alpha) - 1], -1)
    return float(np.linalg.eigvalsh(T)[-1])
