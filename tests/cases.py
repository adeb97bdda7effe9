"""Shared parity cases: each returns (ProblemSetup for the CUDA path, OracleProblem for the CPU
oracle) built from the same reference-style inputs.  Imports of ``oracle`` are confined to
tests (see oracle/__init__.py)."""
import os

import numpy as np

from fea_diffusion_b200.host import MeshTopology, ProblemSetup
from oracle.fea_oracle import OracleProblem, facet_region_vertices, points_on_edge

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
_F = None


def fixtures():
    """The golden arrays by name: tests/golden/fixtures.npz and the reference's displacements (reference_u.npz)."""
    global _F
    if _F is None:
        _F = {}
        for name in ("fixtures.npz", "reference_u.npz"):
            with np.load(os.path.join(ROOT, "tests", "golden", name)) as f:
                _F.update(f)
    return _F


def _override(setup, orc, fixed_sel, loads):
    """Application problem files select regions by coordinate predicates, which the FEAnalysis
    argument surface cannot express: set the Dirichlet mask / load on both objects directly."""
    n_v = len(setup.coors)
    fv_gpu = MeshTopology(setup.conn, n_v).facet_vertices(fixed_sel)
    fv_orc = facet_region_vertices(orc.conn, fixed_sel, n_v)
    assert np.array_equal(fv_gpu, fv_orc)
    setup.sample.fixed[:] = False
    setup.sample.fixed[fv_gpu] = True
    orc.fixed_vertex[:] = False
    orc.fixed_vertex[fv_orc] = True
    setup.sample.rhs[:] = 0
    orc.load[:] = 0
    for verts, mag in loads:
        setup.sample.rhs[verts] += mag
        orc.load[verts] += mag
    return setup, orc


def cantilever(num_steps=11):
    """applications/cantilever/cantilever.py:43-72 (reference)."""
    F = fixtures()
    co, cn = F["cantilever_coors"], F["cantilever_conn"]
    s, o = ProblemSetup(co, cn), OracleProblem(co, cn, num_steps=num_steps)
    return _override(s, o, np.flatnonzero(co[:, 0] < 0.01), [(np.array([3]), (0.0, -1000.0))])


def shearblade(num_steps=11):
    """applications/shearblade/shearblade.py:43-72 (reference)."""
    F = fixtures()
    co, cn = F["shearblade_coors"], F["shearblade_conn"]
    s, o = ProblemSetup(co, cn), OracleProblem(co, cn, num_steps=num_steps)
    return _override(s, o, np.flatnonzero(co[:, 1] > 0.74), [(np.array([1]), (100.0, 3000.0))])


def gusset(num_steps=11):
    """applications/gusset/gusset.py:39-94 (reference); no golden output ships for it."""
    F = fixtures()
    co, cn = F["gusset_coors"], F["gusset_conn"]
    s, o = ProblemSetup(co, cn), OracleProblem(co, cn, num_steps=num_steps)
    n_v = len(co)
    force = facet_region_vertices(o.conn, np.flatnonzero(co[:, 0] > 0.99), n_v)
    force2 = facet_region_vertices(o.conn, points_on_edge(co, (3, 4)), n_v)
    fixed_sel = np.flatnonzero((co[:, 1] < 0.01) | (co[:, 0] < 0.01))
    return _override(s, o, fixed_sel, [(force, (1000.0, 0.0)), (force2, (1000.0, 1000.0))])


def composite_args(well_posed=True):
    """applications/composite/datagenapplication.ipynb:262-264, 300-316 (reference) -- the
    committed condition is singular (two vertex constraints, floating concrete region); the
    well-posed variant constrains the right edge (both regions) and adds an edge force."""
    F = fixtures()
    co, cn = F["composite_coors"], F["composite_conn"]
    concrete = co[co[:, 1] > 0.6875]
    steel = co[co[:, 1] <= 0.6875]
    mats = {(30000, 0.2): concrete, (210000, 0.3): steel}
    if well_posed:
        kw = dict(force_vertex_tags_magnitudes=[(7, (0, -200)), (8, (150, -200))],
                  force_edges_tags_magnitudes=[((9, 10), (-300, 120))],
                  constraints_vertex_tags=[2], constraints_edges_tags=[(4, 5)],
                  material_properties_to_vertices=mats)
    else:
        kw = dict(force_vertex_tags_magnitudes=[(6, (0, -200)), (7, (0, -200)), (8, (0, -200)), (9, (0, -200))],
                  constraints_vertex_tags=[2, 3], material_properties_to_vertices=mats)
    return co, cn, kw


def composite(well_posed=True, num_steps=11):
    co, cn, kw = composite_args(well_posed)
    return ProblemSetup(co, cn, **kw), OracleProblem(co, cn, num_steps=num_steps, **kw)


def quad_plate(nx=24, ny=16, num_steps=5, seed=0):
    """Structured Q1 mesh (unpinned in the reference, F11): jittered grid, left edge fixed,
    point loads on the right edge; some cells deliberately clockwise."""
    rng = np.random.default_rng(seed)
    xs, ys = np.meshgrid(np.linspace(0, 1.5, nx + 1), np.linspace(0, 1.0, ny + 1), indexing="xy")
    co = np.stack([xs.ravel(), ys.ravel()], axis=1)
    inner = (co[:, 0] > 0) & (co[:, 0] < 1.5) & (co[:, 1] > 0) & (co[:, 1] < 1.0)
    co[inner] += 0.25 * (1.0 / max(nx, ny)) * rng.uniform(-1, 1, size=(inner.sum(), 2))
    idx = lambda i, j: j * (nx + 1) + i
    cn = np.array([[idx(i, j), idx(i + 1, j), idx(i + 1, j + 1), idx(i, j + 1)]
                   for j in range(ny) for i in range(nx)], dtype=np.int32)
    flip = rng.random(len(cn)) < 0.3
    cn[flip] = cn[flip][:, [0, 3, 2, 1]]
    # corner tags (1-based): the left edge is the line through vertices idx(0,0) and idx(0,ny)
    kw = dict(force_vertex_tags_magnitudes=[(idx(nx, ny) + 1, (50, -400)), (idx(nx, 0) + 1, (0, 250))],
              constraints_edges_tags=[(idx(0, 0) + 1, idx(0, ny) + 1)],
              youngs_modulus=68900, poisson_ratio=0.33)
    return ProblemSetup(co, cn, **kw), OracleProblem(co, cn, num_steps=num_steps, **kw)
