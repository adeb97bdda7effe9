"""CPU checks of the numpy restatement of the non-nested multigrid path (tests/nonnested_oracle.py): point
location through the grid equals a brute-force search, and the numpy flexible CG converges on a plate whose
coarse level is a coarser mesh of the same geometry."""
import numpy as np

from fea_diffusion_b200.host import ProblemSetup
from fea_diffusion_b200.workload import plate_condition, plate_meshes
from nonnested_oracle import NonNestedMultigrid, locate, locate_brute
from oracle.fea_oracle import fix_orientation


def test_grid_point_location_equals_brute_force():
    (coarse, fine), _, _ = plate_meshes(1, [0.04, 0.02])
    oc = fix_orientation(coarse[0], coarse[1])[0]
    tri, w = locate(fine[0], coarse[0], oc)
    tb, wb = locate_brute(fine[0], coarse[0], oc)
    assert (tri >= 0).all()
    assert np.array_equal(tri, tb) and np.array_equal(w, wb)
    # a vertex pushed out of the domain by more than the tolerance is found by neither
    far = np.vstack([fine[0], [[5.0, 5.0]]])
    assert locate(far, coarse[0], oc)[0][-1] == -1 and locate_brute(far, coarse[0], oc)[0][-1] == -1


def test_nonnested_fcg_converges_on_a_plate():
    meshes, ptags, ltags = plate_meshes(1, [0.04, 0.02])
    kw = plate_condition(ptags, ltags)
    levels = []
    for coors, conn in meshes:
        s = ProblemSetup(coors, conn, **kw).sample
        levels.append((s.coors, s.conn, s.cell_region, s.D, s.fixed))
    mg = NonNestedMultigrid(levels)
    s = ProblemSetup(meshes[-1][0], meshes[-1][1], **kw).sample
    f = s.rhs[~s.fixed].reshape(-1)
    u, it = mg.solve(f, rtol=1e-8, max_iter=100)
    K = mg.K[-1]
    assert np.linalg.norm(f - K @ u) <= 1e-6 * np.linalg.norm(f)
    assert it < 100
