"""numpy/scipy restatement of the non-nested multigrid path of ``fea_batch_set_coarse_meshes`` (TEST
INFRASTRUCTURE; DESIGN.md section 3.10).

Point location with the device's rule and rounding (edge functions and barycentric weights op by op, no
FMA; edge-inclusive; lowest-index containing triangle; else the nearest triangle within 1e-10 x the
longest bounding-box side, weights clamped to [0, 1] and renormalised), the prolongation P between
consecutive levels, rediscretised coarse operators from the oracle assembly, and the Chebyshev V-cycle /
flexible CG of ``oracle.multigrid.Multigrid`` on that hierarchy.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle.fea_oracle import assemble_csr, element_stiffness, equation_map, fix_orientation
from oracle.multigrid import Multigrid, _block_inverse, _lanczos_lmax, block_scaling


def _edge(ax, ay, bx, by, px, py):
    return (bx - ax) * (py - ay) - (by - ay) * (px - ax)


def _seg_d2(ax, ay, bx, by, px, py):
    abx, aby = bx - ax, by - ay
    apx, apy = px - ax, py - ay
    ll = abx * abx + aby * aby
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(ll > 0, (apx * abx + apy * aby) / np.where(ll > 0, ll, 1.0), 0.0)
    t = np.minimum(np.maximum(t, 0.0), 1.0)
    dx, dy = apx - t * abx, apy - t * aby
    return dx * dx + dy * dy


def _pairs_eval(xyf, xyc, conn, v, t):
    """edge functions, containment and squared distance of (vertex v, triangle t) pairs"""
    p = xyf[v]
    a, b, c = xyc[conn[t, 0]], xyc[conn[t, 1]], xyc[conn[t, 2]]
    e0 = _edge(a[:, 0], a[:, 1], b[:, 0], b[:, 1], p[:, 0], p[:, 1])
    e1 = _edge(b[:, 0], b[:, 1], c[:, 0], c[:, 1], p[:, 0], p[:, 1])
    e2 = _edge(c[:, 0], c[:, 1], a[:, 0], a[:, 1], p[:, 0], p[:, 1])
    inside = ((e0 >= 0) & (e1 >= 0) & (e2 >= 0)) | ((e0 <= 0) & (e1 <= 0) & (e2 <= 0))
    d2 = np.minimum(_seg_d2(a[:, 0], a[:, 1], b[:, 0], b[:, 1], p[:, 0], p[:, 1]),
                    np.minimum(_seg_d2(b[:, 0], b[:, 1], c[:, 0], c[:, 1], p[:, 0], p[:, 1]),
                               _seg_d2(c[:, 0], c[:, 1], a[:, 0], a[:, 1], p[:, 0], p[:, 1])))
    return inside, d2


def _pick(nf, v, t, inside, d2, tol2):
    """per vertex: lowest containing triangle, else the nearest (ties: lowest index) within tol; -1 = none"""
    tri = np.full(nf, -1, np.int64)
    if len(v):
        o = np.lexsort((t, ~inside, v))         # per vertex: containing first, then ascending triangle
        first = np.r_[True, v[o][1:] != v[o][:-1]]
        vi, ti, ii = v[o][first], t[o][first], inside[o][first]
        tri[vi[ii]] = ti[ii]
        o = np.lexsort((t, d2, v))              # nearest, ties to the lowest index
        first = np.r_[True, v[o][1:] != v[o][:-1]]
        vn, tn, dn = v[o][first], t[o][first], d2[o][first]
        near = (tri[vn] < 0) & (dn <= tol2)
        tri[vn[near]] = tn[near]
    return tri


def _weights(xyf, xyc, conn, tri, inside):
    p = xyf
    a, b, c = xyc[conn[tri, 0]], xyc[conn[tri, 1]], xyc[conn[tri, 2]]
    e0 = _edge(a[:, 0], a[:, 1], b[:, 0], b[:, 1], p[:, 0], p[:, 1])
    e1 = _edge(b[:, 0], b[:, 1], c[:, 0], c[:, 1], p[:, 0], p[:, 1])
    e2 = _edge(c[:, 0], c[:, 1], a[:, 0], a[:, 1], p[:, 0], p[:, 1])
    s = (e0 + e1) + e2
    w = np.stack([e1 / s, e2 / s, e0 / s], 1)
    wc = np.minimum(np.maximum(w, 0.0), 1.0)
    wc = wc / ((wc[:, 0:1] + wc[:, 1:2]) + wc[:, 2:3])
    return np.where(inside[:, None], w, wc)


def _tolerance(xyc):
    ext = xyc.max(0) - xyc.min(0)
    return 1e-10 * float(max(ext[0], ext[1]))


def locate_brute(xyf, xyc, conn) -> Tuple[np.ndarray, np.ndarray]:
    """(triangle per fine vertex or -1 if farther than the tolerance, (n_f, 3) weights of its vertices), by
    testing every triangle: for small meshes."""
    xyf, xyc, conn = np.asarray(xyf, float), np.asarray(xyc, float), np.asarray(conn, np.int64)
    tol = _tolerance(xyc)
    nf, nc = len(xyf), len(conn)
    v, t = np.repeat(np.arange(nf), nc), np.tile(np.arange(nc), nf)
    inside, d2 = _pairs_eval(xyf, xyc, conn, v, t)
    tri = _pick(nf, v, t, inside, d2, tol * tol)
    return tri, _finish(xyf, xyc, conn, tri, v, t, inside)


def _finish(xyf, xyc, conn, tri, v, t, inside):
    contained = np.zeros(len(xyf), bool)
    contained[v[inside]] = True
    w = np.zeros((len(xyf), 3))
    ok = tri >= 0
    w[ok] = _weights(xyf[ok], xyc, conn, tri[ok], contained[ok])
    return w


def locate(xyf, xyc, conn) -> Tuple[np.ndarray, np.ndarray]:
    """``locate_brute``'s result through a uniform grid of about one cell per triangle (what the device does)."""
    xyf, xyc, conn = np.asarray(xyf, float), np.asarray(xyc, float), np.asarray(conn, np.int64)
    tol = _tolerance(xyc)
    lo, hi = xyc.min(0), xyc.max(0)
    W, H = hi - lo
    hg = np.sqrt(max(W * H, 1e-300) / max(len(conn), 1))
    nx = max(1, int(min(np.ceil(W / hg), 4096))) if W > 0 else 1
    ny = max(1, int(min(np.ceil(H / hg), 4096))) if H > 0 else 1
    inv = np.array([nx / W if W > 0 else 0.0, ny / H if H > 0 else 0.0])
    n = np.array([nx, ny])

    def bins(q):
        return np.clip(np.floor((q - lo) * inv), 0, n - 1).astype(np.int64)

    P = xyc[conn]
    b0, b1 = bins(P.min(1) - tol), bins(P.max(1) + tol)
    cx, cy = b1[:, 0] - b0[:, 0] + 1, b1[:, 1] - b0[:, 1] + 1    # grid cells covered by each grown bounding box
    tris = np.repeat(np.arange(len(conn)), cx * cy)
    k = np.arange(len(tris)) - np.repeat(np.concatenate([[0], np.cumsum(cx * cy)[:-1]]), cx * cy)
    cells = (b0[tris, 1] + k // cx[tris]) * nx + b0[tris, 0] + k % cx[tris]
    o = np.argsort(cells, kind="stable")
    cells, tris = cells[o], tris[o]
    ptr = np.searchsorted(cells, np.arange(nx * ny + 1))
    bf = bins(xyf)
    cf = bf[:, 1] * nx + bf[:, 0]
    cnt = ptr[cf + 1] - ptr[cf]
    v = np.repeat(np.arange(len(xyf)), cnt)
    start = np.repeat(ptr[cf] - np.concatenate([[0], np.cumsum(cnt)[:-1]]), cnt)
    t = tris[start + np.arange(len(v))]
    inside, d2 = _pairs_eval(xyf, xyc, conn, v, t)
    tri = _pick(len(xyf), v, t, inside, d2, tol * tol)
    return tri, _finish(xyf, xyc, conn, tri, v, t, inside)


def prolongation(conn_c, tri, w, n_coarse) -> sp.csr_matrix:
    """P over all DOFs (2 n_fine x 2 n_coarse): each component from the located triangle's vertices, zero weights
    dropped."""
    nf = len(tri)
    f = np.repeat(np.arange(nf), 3)
    par = np.asarray(conn_c, np.int64)[np.maximum(tri, 0)].reshape(-1)
    wv = w.reshape(-1)
    keep = (np.repeat(tri, 3) >= 0) & (wv != 0.0)
    rows = np.concatenate([2 * f[keep], 2 * f[keep] + 1])
    cols = np.concatenate([2 * par[keep], 2 * par[keep] + 1])
    return sp.csr_matrix((np.concatenate([wv[keep], wv[keep]]), (rows, cols)), shape=(2 * nf, 2 * n_coarse))


class NonNestedMultigrid(Multigrid):
    """Hierarchy of meshes of one domain, coarsest first: each (coors, conn as given, cell_region, D per region,
    fixed vertices).  Operators are rediscretised on every level; P by point location."""

    def __init__(self, meshes: Sequence, degree: int = 3, lanczos_steps: int = 20):
        self.levels, self.degree = len(meshes) - 1, degree
        self.oriented, self.fixed, self.K, self.P, self.tri = [], [], [], [None], [None]
        for coors, conn, creg, D, fixed in meshes:
            coors = np.asarray(coors, float)
            creg = np.asarray(creg)
            oc = fix_orientation(coors, conn)[0]
            ke = element_stiffness(coors, oc, np.asarray(D)[np.maximum(creg, 0)])
            ke[creg < 0] = 0.0
            self.K.append(assemble_csr(len(coors), oc, ke, creg, np.asarray(fixed, bool)))
            self.oriented.append(oc)
            self.fixed.append(np.asarray(fixed, bool))
        for l in range(1, len(meshes)):
            tri, w = locate(meshes[l][0], meshes[l - 1][0], self.oriented[l - 1])
            if (tri < 0).any():
                raise ValueError("level %d: vertex %d outside level %d" % (l, int(np.flatnonzero(tri < 0)[0]), l - 1))
            eq_f, _ = equation_map(self.fixed[l])
            eq_c, _ = equation_map(self.fixed[l - 1])
            P = prolongation(self.oriented[l - 1], tri, w, len(meshes[l - 1][0]))
            self.P.append(P[eq_f >= 0][:, eq_c >= 0].tocsr())
            self.tri.append(tri)
        self.S = [block_scaling(K) for K in self.K]
        self.Kh = [(S.T @ K @ S).tocsr() for S, K in zip(self.S, self.K)]
        self.Ph = [None] + [(_block_inverse(self.S[l]) @ self.P[l] @ self.S[l - 1]).tocsr() for l in range(1, self.levels + 1)]
        self.lmax = [_lanczos_lmax(A, lanczos_steps) for A in self.Kh]
        self.coarse = spla.splu(self.Kh[0].tocsc())
