"""numpy/scipy restatement of the grid hierarchy of ``fea_batch_set_grid_hierarchy`` (TEST INFRASTRUCTURE;
DESIGN.md section 3.12).

Nested background grids over the mesh's bounding box, point location of the mesh's vertices in the finest
grid (``nonnested_oracle.locate``, the device's rule and rounding), analytic grid-to-grid weights 1 and 1/2,
pruning to the vertices that active vertices of the next finer level reach, and Galerkin operators
K_(l-1) = P^T K_l P.  The V-cycle and flexible CG are those of ``oracle.multigrid.Multigrid``.
"""
from __future__ import annotations

from typing import List, Tuple

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from nonnested_oracle import locate
from oracle.fea_oracle import assemble_csr, element_stiffness, equation_map, fix_orientation
from oracle.multigrid import Multigrid, _block_inverse, _lanczos_lmax, block_scaling

CHUNK = 1024   # items a device thread sums in order, before one thread sums the chunk sums in order


def _ordered_sum(a: np.ndarray) -> float:
    """The device's fixed-order sum: chunks of CHUNK summed left to right, then the chunk sums (cumsum is
    sequential)."""
    pad = np.zeros(-len(a) % CHUNK)
    c = np.concatenate([a, pad]).reshape(-1, CHUNK)
    part = np.cumsum(c, axis=1)[:, -1] if len(c) else np.zeros(1)
    return float(np.cumsum(part)[-1])


def grid_spacing(coors, oriented) -> float:
    """h = sqrt(2 A / n_cells), A the summed cell area (twice-areas rounded op by op, as the device)."""
    x, y = coors[oriented, 0], coors[oriented, 1]
    a2 = np.zeros(len(oriented))
    for a in range(3):
        n = (a + 1) % 3
        a2 = a2 + (x[:, a] * y[:, n] - x[:, n] * y[:, a])
    A2 = _ordered_sum(np.abs(a2))
    return float(np.sqrt(A2 / len(oriented)))


class Grid:
    """Grid with nx x ny squares of side H from (x0, y0); vertex (i, j) is j * (nx + 1) + i, square (i, j)
    holds triangles 2s = (v(i,j), v(i+1,j), v(i+1,j+1)) and 2s+1 = (v(i,j), v(i+1,j+1), v(i,j+1)), s = j nx + i."""

    def __init__(self, x0, y0, H, nx, ny):
        self.x0, self.y0, self.H, self.nx, self.ny = x0, y0, H, nx, ny
        i, j = np.meshgrid(np.arange(nx + 1, dtype=float), np.arange(ny + 1, dtype=float))
        self.xy = np.stack([x0 + i.ravel() * H, y0 + j.ravel() * H], 1)
        si, sj = np.meshgrid(np.arange(nx), np.arange(ny))
        si, sj = si.ravel(), sj.ravel()
        v = lambda a, b: b * (nx + 1) + a
        t0 = np.stack([v(si, sj), v(si + 1, sj), v(si + 1, sj + 1)], 1)
        t1 = np.stack([v(si, sj), v(si + 1, sj + 1), v(si, sj + 1)], 1)
        self.conn = np.stack([t0, t1], 1).reshape(-1, 3)


def grids(coors, conn, levels: int) -> List[Grid]:
    """The grids of coarse levels 0..levels-1, coarsest first."""
    coors = np.asarray(coors, float)
    oc = fix_orientation(coors, conn)[0]
    h = grid_spacing(coors, oc)
    lo, hi = coors.min(0), coors.max(0)
    ext = hi - lo
    tol = 1e-10 * float(max(ext[0], ext[1]))
    x0, y0 = lo[0] - tol, lo[1] - tol
    x1, y1 = hi[0] + tol, hi[1] + tol
    H0 = (2.0 * h) * float(2 ** (levels - 1))
    n = []
    for a0, a1 in ((x0, x1), (y0, y1)):
        k = max(1, int(np.ceil((a1 - a0) / H0)))
        while a0 + k * H0 < a1:
            k += 1
        n.append(k)
    return [Grid(x0, y0, H0 / float(2 ** l), n[0] << l, n[1] << l) for l in range(levels)]


def grid_prolongation(f: Grid, c: Grid) -> sp.csr_matrix:
    """Scalar P (n_f x n_c) of the red refinement f of c: weight 1 at even (i, j), 1/2 from the two ends of
    the coarse edge (horizontal, vertical or the diagonal (i, j)-(i+1, j+1)) otherwise."""
    i, j = np.meshgrid(np.arange(f.nx + 1), np.arange(f.ny + 1))
    i, j = i.ravel(), j.ravel()
    rows = np.arange(len(i))
    cv = lambda a, b: b * (c.nx + 1) + a
    a0, b0 = i // 2, j // 2
    a1, b1 = (i + 1) // 2, (j + 1) // 2
    same = (i % 2 == 0) & (j % 2 == 0)
    r = np.concatenate([rows[same], rows[~same], rows[~same]])
    col = np.concatenate([cv(a0, b0)[same], cv(a0, b0)[~same], cv(a1, b1)[~same]])
    w = np.concatenate([np.ones(same.sum()), np.full(2 * (~same).sum(), 0.5)])
    return sp.csr_matrix((w, (r, col)), shape=(len(i), len(c.xy)))


def _dofs(P: sp.csr_matrix) -> sp.csr_matrix:
    return sp.kron(P, sp.eye(2), format="csr")


class GridMultigrid(Multigrid):
    """Grid hierarchy of one mesh (coors, conn as given, cell_region, D per region, fixed vertices): coarse
    levels 0..levels-1 are pruned grids with Galerkin operators, level ``levels`` the mesh."""

    def __init__(self, coors, conn, cell_region, D, fixed, levels: int, degree: int = 3, lanczos_steps: int = 20):
        coors = np.asarray(coors, float)
        fixed = np.asarray(fixed, bool)
        creg = np.asarray(cell_region)
        self.levels, self.degree = levels, degree
        oc = fix_orientation(coors, conn)[0]
        ke = element_stiffness(coors, oc, np.asarray(D)[np.maximum(creg, 0)])
        ke[creg < 0] = 0.0
        K_mesh = assemble_csr(len(coors), oc, ke, creg, fixed)
        self.grids = grids(coors, conn, levels)
        # scalar P over all vertices, finest first: mesh -> finest grid by point location, then analytic
        g = self.grids[-1]
        tri, w = locate(coors, g.xy, g.conn)
        if (tri < 0).any():
            raise ValueError("a mesh vertex lies outside the grid")
        keep = w.reshape(-1) != 0.0
        rows = np.repeat(np.arange(len(coors)), 3)[keep]
        cols = g.conn[tri].reshape(-1)[keep]
        Pfull = [None] * (levels + 1)
        Pfull[levels] = sp.csr_matrix((w.reshape(-1)[keep], (rows, cols)), shape=(len(coors), len(g.xy)))
        for l in range(levels - 1, 0, -1):
            Pfull[l] = grid_prolongation(self.grids[l], self.grids[l - 1])
        # pruning: active vertices reach their parents; kept cells have an active vertex
        active = [None] * (levels + 1)
        active[levels] = ~fixed
        self.kept_v, self.kept_c = [None] * levels, [None] * levels
        for l in range(levels - 1, -1, -1):
            Pa = Pfull[l + 1][active[l + 1]]
            a = np.zeros(Pa.shape[1], bool)
            a[Pa.indices[Pa.data != 0.0]] = True
            cells = a[self.grids[l].conn].any(1)
            kv = np.zeros(len(a), bool)
            kv[self.grids[l].conn[cells].reshape(-1)] = True
            self.kept_v[l], self.kept_c[l] = np.flatnonzero(kv), np.flatnonzero(cells)
            active[l] = a
        # the level meshes in kept numbering, their fixed masks, and P between kept vertices
        self.coors, self.conn, self.fixed = [], [], []
        for l in range(levels):
            kv = self.kept_v[l]
            new = np.full(len(self.grids[l].xy), -1, np.int64)
            new[kv] = np.arange(len(kv))
            self.coors.append(self.grids[l].xy[kv])
            self.conn.append(new[self.grids[l].conn[self.kept_c[l]]])
            self.fixed.append(~active[l][kv])
        self.coors.append(coors)
        self.conn.append(oc)
        self.fixed.append(fixed)
        self.P_all = [None]   # scalar P over kept vertices of both levels
        for l in range(1, levels + 1):
            rows_kept = self.kept_v[l] if l < levels else np.arange(len(coors))
            self.P_all.append(Pfull[l][rows_kept][:, self.kept_v[l - 1]].tocsr())
        self.P = [None]
        for l in range(1, levels + 1):
            eq_f, _ = equation_map(self.fixed[l])
            eq_c, _ = equation_map(self.fixed[l - 1])
            self.P.append(_dofs(self.P_all[l])[eq_f >= 0][:, eq_c >= 0].tocsr())
        self.K = [None] * (levels + 1)
        self.K[levels] = K_mesh
        for l in range(levels, 0, -1):
            self.K[l - 1] = (self.P[l].T @ self.K[l] @ self.P[l]).tocsr()
        self.S = [block_scaling(K) for K in self.K]
        self.Kh = [(S.T @ K @ S).tocsr() for S, K in zip(self.S, self.K)]
        self.Ph = [None] + [(_block_inverse(self.S[l]) @ self.P[l] @ self.S[l - 1]).tocsr() for l in range(1, levels + 1)]
        self.lmax = [_lanczos_lmax(A, lanczos_steps) for A in self.Kh]
        self.coarse = spla.splu(self.Kh[0].tocsc())

    def row_lengths(self) -> List[int]:
        """Largest number of 2x2 blocks in a row (the diagonal included) of every level."""
        return [int(np.diff(K.indptr).max()) // 2 for K in self.K]

    def energy_contraction(self, seed: int = 1) -> float:
        """||x - M K x||_K / ||x||_K for a random x on the finest level (exact coarse solve)."""
        K = self.K[self.levels]
        x = np.random.default_rng(seed).standard_normal(K.shape[0])
        e = x - self.apply_unscaled(K @ x)
        return float(np.sqrt(e @ (K @ e)) / np.sqrt(x @ (K @ x)))
