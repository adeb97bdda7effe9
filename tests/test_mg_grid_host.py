"""CPU checks of the numpy restatement of the grid hierarchy (tests/grid_oracle.py): nested grids, P reproduces
linear fields, symmetric Galerkin levels with positive definite diagonal blocks, row lengths within the
adjacency cap, and the V-cycle's energy-norm contraction with an exact coarse solve."""
import numpy as np
import pytest

from fea_diffusion_b200.host import ProblemSetup
from fea_diffusion_b200.workload import jittered_case, plate_condition, plate_meshes
from grid_oracle import GridMultigrid, grids
from oracle.fea_oracle import equation_map

MAX_ADJ = 64   # kMaxAdj: a row holds at most 63 neighbours besides the diagonal


def plate_with_holes():
    (mesh,), ptags, ltags = plate_meshes(1, [0.02])
    return ProblemSetup(mesh[0], mesh[1], **plate_condition(ptags, ltags)).sample


def two_material_plate():
    s = plate_with_holes()
    xy = s.coors[np.asarray(s.conn)].mean(1)
    creg = (xy[:, 0] > np.median(xy[:, 0])).astype(np.int8)
    D = np.stack([s.D[0], 20.0 * s.D[0]])
    return s.__class__(s.coors, s.conn, creg, D, s.fixed, s.rhs)


CASES = {
    "plate_with_holes": (plate_with_holes, 2),
    "two_material_plate": (two_material_plate, 2),
    "jittered_cantilever_l2": (lambda: jittered_case("cantilever", 2)[0], 2),
}


@pytest.fixture(scope="module", params=sorted(CASES))
def case(request):
    make, levels = CASES[request.param]
    s = make()
    return request.param, s, GridMultigrid(s.coors, s.conn, s.cell_region, s.D, s.fixed, levels)


def test_grids_are_nested_bit_for_bit():
    s = plate_with_holes()
    g = grids(s.coors, s.conn, 3)
    for c, f in zip(g[:-1], g[1:]):
        assert f.nx == 2 * c.nx and f.ny == 2 * c.ny and f.H * 2.0 == c.H
        even = f.xy.reshape(f.ny + 1, f.nx + 1, 2)[::2, ::2].reshape(-1, 2)
        assert np.array_equal(even, c.xy)
    lo, hi = s.coors.min(0), s.coors.max(0)
    assert (g[0].xy.min(0) < lo).all() and (g[0].xy.max(0) >= hi).all()


def test_prolongation_reproduces_linear_fields(case):
    name, s, mg = case
    for l in range(1, mg.levels + 1):
        P = mg.P_all[l]
        # every parent of an active fine vertex is kept, so its row is complete
        act = ~np.asarray(mg.fixed[l], bool)
        assert np.abs(np.asarray(P.sum(axis=1)).ravel()[act] - 1.0).max() <= 1e-14
        for a, b, c in ((1.0, 0.0, 0.0), (0.3, 2.0, -1.5)):
            gc = a + b * mg.coors[l - 1][:, 0] + c * mg.coors[l - 1][:, 1]
            gf = a + b * mg.coors[l][:, 0] + c * mg.coors[l][:, 1]
            assert np.abs((P @ gc - gf)[act]).max() <= 1e-12 * max(1.0, np.abs(gf).max())


def test_galerkin_levels_are_spd_and_within_the_cap(case):
    name, s, mg = case
    lengths = mg.row_lengths()
    print("%s: level vertices %s, active DOFs %s, max blocks per row %s, contraction %.3f" % (
        name, [len(c) for c in mg.coors], [K.shape[0] for K in mg.K], lengths, mg.energy_contraction()))
    assert max(lengths[:-1]) < MAX_ADJ
    for l in range(mg.levels):
        K = mg.K[l]
        assert abs(K - K.T).max() <= 1e-12 * abs(K).max()
        d = K.diagonal()
        dc = np.asarray(K[np.arange(0, K.shape[0], 2), np.arange(1, K.shape[0], 2)]).ravel()
        assert (d > 0).all() and (d[0::2] * d[1::2] - dc * dc > 0).all()
        # every kept active vertex of a coarse level has a row, and every row a non-zero weight from below
        eq, n = equation_map(mg.fixed[l])
        assert n == K.shape[0] and (np.diff(mg.P[l + 1].tocsc().indptr) > 0).all()


def test_vcycle_contracts_the_energy_norm(case):
    """At most 0.5 with an exact coarse solve (the coarse meshes of DESIGN.md section 3.10 give 0.27)."""
    name, s, mg = case
    assert mg.energy_contraction() <= 0.5


def test_fcg_converges_on_the_plate_with_holes():
    s = plate_with_holes()
    mg = GridMultigrid(s.coors, s.conn, s.cell_region, s.D, s.fixed, 3)
    f = s.rhs[~s.fixed.astype(bool)].reshape(-1)
    u, it = mg.solve(f, rtol=1e-10, max_iter=100)
    assert np.linalg.norm(f - mg.K[-1] @ u) <= 1e-9 * np.linalg.norm(f)
    assert it <= 60   # 44 with the exact coarse solve, where a random vector contracts by 0.24 per V-cycle
