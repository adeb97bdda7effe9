"""Multigrid-preconditioned solve of uniformly refined meshes (fea_batch_set_refinement): hierarchy checks,
Galerkin operators against numpy's P^T K P, V-cycle contraction, parity with direct solves, outer iteration
counts, determinism and the outputs downstream of the solve."""
import os

import numpy as np
import pytest

import cases
from fea_diffusion_b200 import Context, FeaError, pack
from fea_diffusion_b200._capi import SAMPLE_CONVERGED
from fea_diffusion_b200.solver import Sample
from fea_diffusion_b200.workload import large_case
from oracle.multigrid import Multigrid

pytestmark = pytest.mark.gpu

BAD_ARG, MESH_ERROR = 1, 5


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


def cantilever(levels):
    setup, _ = large_case("cantilever", levels)
    return setup.sample


def with_mesh(s, coors, conn):
    return Sample(coors, conn, s.cell_region, s.D, s.fixed, s.rhs)


def set_refinement_code(ctx, samples, levels):
    with ctx.create_batch(pack(samples)) as b:
        try:
            b.set_refinement(levels)
        except FeaError as e:
            return e.code
    return 0


@pytest.mark.parametrize("levels", [1, 2, 3, 4])
def test_set_refinement_accepts_uniform_refinements(ctx, levels):
    assert set_refinement_code(ctx, [cantilever(levels)], levels) == 0


def test_set_refinement_rejects_what_is_not_such_a_refinement(ctx):
    s = cantilever(2)
    n0 = len(cases.fixtures()["cantilever_coors"])
    nc = len(s.conn) // 4
    moved = s.coors.copy()
    moved[len(moved) - 1, 0] = np.nextafter(moved[len(moved) - 1, 0], np.inf)   # one midpoint, one ulp
    assert set_refinement_code(ctx, [with_mesh(s, moved, s.conn)], 2) == MESH_ERROR
    swapped = s.conn.copy()
    swapped[[5, 5 + nc]] = swapped[[5 + nc, 5]]                                   # two children of cell 5
    assert set_refinement_code(ctx, [with_mesh(s, s.coors, swapped)], 2) == MESH_ERROR
    assert set_refinement_code(ctx, [s], 3) == MESH_ERROR                         # one level too many
    assert n0 < len(s.coors)


def test_set_refinement_rejects_a_vertex_that_is_no_midpoint(ctx):
    """The coarse mesh's last vertex belongs to no cell: after refinement it sits where the midpoints
    start, and it is the midpoint of no edge.  The block-Jacobi path solves such a mesh; the hierarchy
    cannot be derived from it."""
    from fea_diffusion_b200 import ProblemSetup
    from fea_diffusion_b200.workload import refine_uniform
    F = cases.fixtures()
    c0 = np.vstack([F["cantilever_coors"], [[2.0, 2.0]]])
    co, cn = refine_uniform(c0, F["cantilever_conn"], 2)
    s = ProblemSetup(co, cn).sample
    s.fixed[:] = co[:, 0] < 0.01
    s.fixed[len(c0) - 1] = True
    s.rhs[:] = 0
    s.rhs[3] = (0.0, -1000.0)
    assert set_refinement_code(ctx, [s], 2) == MESH_ERROR
    with ctx.create_batch(pack([s])) as b:      # the batch itself is fine for the block-Jacobi path
        r = b.assemble().solve(1e-10, 200000).download()
    assert r.status[0] == SAMPLE_CONVERGED


def test_set_refinement_bad_arguments(ctx):
    s = cantilever(1)
    assert set_refinement_code(ctx, [s, s], 1) == BAD_ARG
    xy = np.array([[0, 0], [1, 0], [2, 0], [0, 1], [1, 1], [2, 1]], np.float64)
    q = Sample(xy, np.array([[0, 1, 4, 3], [1, 2, 5, 4]], np.int32), np.zeros(2, np.int8), s.D[:1],
               np.array([1, 0, 0, 1, 0, 0], np.uint8), np.zeros((6, 2)))
    assert set_refinement_code(ctx, [q], 1) == BAD_ARG
    assert set_refinement_code(ctx, [s], 0) == BAD_ARG
    with ctx.create_batch(pack([s])) as b:
        b.assemble()
        with pytest.raises(FeaError):
            b.set_refinement(1)


@pytest.fixture(scope="module")
def l2(ctx):
    s = cantilever(2)
    mg = Multigrid(s.coors, s.conn, s.cell_region, s.D, s.fixed, 2)
    b = ctx.create_batch(pack([s])).set_refinement(2).assemble()
    yield s, mg, b
    b.destroy()


def test_galerkin_operators_match_numpy(l2):
    s, mg, b = l2
    levels = b.mg_levels()
    assert len(levels) == 3
    for l in range(3):
        Kd, Ko = b.level_csr(l), mg.K[l]
        assert Kd.shape == Ko.shape and levels[l]["n_active_dofs"] == Ko.shape[0]
        assert abs(Kd - Ko).max() <= 1e-12 * abs(Ko).max()
        pattern = Ko.copy()
        pattern.data[:] = 1.0
        outside = Kd - Kd.multiply(pattern)
        assert np.count_nonzero(outside.data) == 0
        assert 1.9 < levels[l]["lambda_max"] < 2.6
    ref = mg.galerkin_reference(0)
    assert abs(b.level_csr(0) - ref).max() <= 1e-12 * abs(ref).max()


def test_vcycle_contracts_the_error(l2):
    """||x - M K x||_K <= c ||x||_K for random x: 0.268 measured on a B200 (the numpy V-cycle with an exact
    coarse solve gives 0.268 as well, although the device's coarse solve stops at rtol 1e-4)."""
    s, mg, b = l2
    K = b.csr(0)
    x = np.random.default_rng(1).standard_normal(K.shape[0])
    e = x - b.mg_apply(K @ x)
    ratio = np.sqrt(e @ (K @ e)) / np.sqrt(x @ (K @ x))
    eo = x - mg.apply_unscaled(K @ x)
    print("V-cycle energy contraction: device", ratio, "numpy, exact coarse solve", np.sqrt(eo @ (K @ eo)) / np.sqrt(x @ (K @ x)))
    assert ratio <= 0.3


@pytest.mark.parametrize("levels", [2, 3])
def test_cantilever_matches_the_direct_solve(ctx, levels):
    import scipy.sparse.linalg as spla
    s = cantilever(levels)
    mg = Multigrid(s.coors, s.conn, s.cell_region, s.D, s.fixed, levels)
    act = ~s.fixed.astype(bool)
    u = np.zeros_like(s.rhs)
    u[act] = spla.spsolve(mg.K[levels].tocsc(), s.rhs[act].reshape(-1)).reshape(-1, 2)
    with ctx.create_batch(pack([s])) as b:
        r = b.set_refinement(levels).assemble().solve(1e-10, 200).download()
    assert r.status[0] == SAMPLE_CONVERGED
    assert np.linalg.norm(r.u - u) / np.linalg.norm(u) <= 1e-8


@pytest.mark.parametrize("name,level", [("cantilever", 4), ("gusset", 3)])
def test_config3_meshes_match_the_stored_sparse_lu_solution(ctx, name, level):
    ref = np.load(os.path.join(cases.ROOT, "tests", "golden", "c3_lu.npz"))
    setup, n0 = large_case(name, level)
    smp = setup.sample
    with ctx.create_batch(pack([smp])) as b:
        r = b.set_refinement(level).assemble().solve(1e-10, 200).download()
        st = b.stats()
        K = b.csr(0)
    assert r.status[0] == SAMPLE_CONVERGED and st["iterations"] <= 40
    g = ref["%s_L%d_u_coarse" % (name, level)]
    err = float(np.linalg.norm(r.u[:n0] - g) / np.linalg.norm(g))
    assert err <= 1e-8, err
    # relres is the TRUE residual in the block-Jacobi-scaled norm
    act = ~smp.fixed.astype(bool)
    f = smp.rhs[act].reshape(-1)
    res = f - K @ r.u[act].reshape(-1)
    from oracle.multigrid import block_scaling
    S = block_scaling(K)
    true_rel = np.linalg.norm(S.T @ res) / np.linalg.norm(S.T @ f)
    assert abs(r.relres[0] - true_rel) <= 0.25 * true_rel


@pytest.mark.parametrize("name,level", [("cantilever", 1), ("cantilever", 2), ("cantilever", 3), ("cantilever", 4),
                                        ("gusset", 1), ("gusset", 2), ("gusset", 3)])
def test_outer_iterations_stay_flat_under_refinement(ctx, name, level):
    setup, _ = large_case(name, level)
    with ctx.create_batch(pack([setup.sample])) as b:
        r = b.set_refinement(level).assemble().solve(1e-10, 200).download()
        st = b.stats()
        lv = b.mg_levels()
    print(name, level, st["iterations"], "%.2f ms" % st["solve_ms"], [round(x["vcycle_ms"], 2) for x in lv])
    assert r.status[0] == SAMPLE_CONVERGED and 1 <= st["iterations"] <= 40 and r.iters[0] == st["iterations"]


def test_deterministic_and_downstream_outputs(ctx):
    s = cantilever(3)
    lo, hi = s.coors.min(0), s.coors.max(0)
    size = 256
    scale = (size - 1) / (hi - lo).max()
    aff = np.array([[scale, -scale * lo[0], scale, -scale * lo[1]]])
    out = []
    for mg in (True, True, False):
        with ctx.create_batch(pack([s])) as b:
            if mg:
                b.set_refinement(3)
            r = b.assemble().solve(1e-10, 200000).rasterize(size, aff, 1.0).download(images=True)
            strain, stress = b.cell_strain_stress()
        out.append((r, strain))
    (a, sa), (b2, sb), (c, sc) = out
    assert np.array_equal(a.u, b2.u) and np.array_equal(a.images, b2.images) and np.array_equal(sa, sb)
    assert np.abs(a.images.astype(int) - c.images.astype(int)).max() <= 1
    assert np.linalg.norm(a.u - c.u) / np.linalg.norm(c.u) <= 1e-8
    assert np.allclose(a.ranges, c.ranges, rtol=1e-8, atol=0)
    assert np.linalg.norm(sa - sc) / np.linalg.norm(sc) <= 1e-7
