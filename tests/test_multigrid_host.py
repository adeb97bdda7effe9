"""CPU checks of the numpy restatement of the multigrid path (oracle/multigrid.py) that the GPU tests
compare against: the cell-by-cell Galerkin sum equals P^T K P, and the Chebyshev V-cycle keeps the
outer flexible-CG iteration count flat under refinement."""
import numpy as np
import pytest
import scipy.sparse.linalg as spla

from fea_diffusion_b200.workload import large_case
from oracle.multigrid import Multigrid, hierarchy


def problem(name, levels):
    setup, n0 = large_case(name, levels)
    s = setup.sample
    return s, n0, Multigrid(s.coors, s.conn, s.cell_region, s.D, s.fixed, levels)


def test_hierarchy_recovers_the_coarse_mesh():
    from fea_diffusion_b200.workload import refine_uniform
    import cases
    F = cases.fixtures()
    co, cn = refine_uniform(F["cantilever_coors"], F["cantilever_conn"], 2)
    conns, pars = hierarchy(cn, 2)
    assert np.array_equal(conns[0], F["cantilever_conn"])
    n1 = int(conns[1].max()) + 1
    mid = pars[2][n1:]
    assert np.array_equal(co[n1:], 0.5 * (co[mid[:, 0]] + co[mid[:, 1]]))


def test_elementwise_galerkin_equals_ptkp_on_cantilever_l2():
    """The fine Dirichlet set (x < 0.01 facets) is not a union of coarse facets here."""
    s, n0, mg = problem("cantilever", 2)
    for l in range(2):
        ref = mg.galerkin_reference(l)
        assert abs(mg.K[l] - ref).max() <= 1e-13 * abs(ref).max()


@pytest.mark.parametrize("levels", [1, 2, 3])
def test_mg_fcg_solves_cantilever_in_few_outer_iterations(levels):
    s, n0, mg = problem("cantilever", levels)
    act = ~s.fixed.astype(bool)
    f = s.rhs[act].reshape(-1)
    u, it = mg.solve(f, 1e-10)
    ud = spla.spsolve(mg.K[levels].tocsc(), f)
    assert it <= 30
    assert np.linalg.norm(u - ud) / np.linalg.norm(ud) <= 1e-8
