"""Multigrid solve of a mesh with no coarse meshes given, from nested background grids with Galerkin operators
(fea_batch_set_grid_hierarchy): the levels and transfers against numpy (tests/grid_oracle.py), determinism,
convergence against block-Jacobi CG and a stored sparse LU solution, load cases, and the return codes."""
import ctypes as C
import os

import numpy as np
import pytest

from fea_diffusion_b200 import Context, FeaError, pack
from fea_diffusion_b200.host import ProblemSetup
from fea_diffusion_b200.solver import PackedConditions, Sample
from fea_diffusion_b200._capi import SAMPLE_BREAKDOWN, SAMPLE_CONVERGED
from fea_diffusion_b200.workload import jittered_case, large_case, plate_condition, plate_meshes
from grid_oracle import GridMultigrid

pytestmark = pytest.mark.gpu

BAD_ARG, BAD_STATE, MESH_ERROR = 1, 4, 5
RTOL, MAX_ITER = 1e-10, 200


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


def plate(h):
    (mesh,), ptags, ltags = plate_meshes(1, [h])
    kw = plate_condition(ptags, ltags)
    return ProblemSetup(mesh[0], mesh[1], **kw).sample, mesh, kw


def rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def with_rhs(s, rhs):
    return Sample(s.coors, s.conn, s.cell_region, s.D, s.fixed, np.ascontiguousarray(rhs))


@pytest.mark.parametrize("name,levels", [("plate-0.01", 2), ("jittered-cantilever-L2", 3)])
def test_levels_and_transfers_match_numpy(ctx, name, levels):
    s = plate(0.01)[0] if name.startswith("plate") else jittered_case("cantilever", 2)[0]
    mg = GridMultigrid(s.coors, s.conn, s.cell_region, s.D, s.fixed, levels)
    with ctx.create_batch(pack([s])) as b:
        b.set_grid_hierarchy(levels).assemble()
        lv = b.mg_levels()
        assert [x["n_vertices"] for x in lv] == [len(c) for c in mg.coors]
        assert [x["n_active_dofs"] for x in lv] == [K.shape[0] for K in mg.K]
        rows = []
        for l in range(levels):
            Kd, Ko = b.level_csr(l), mg.K[l]
            assert Kd.shape == Ko.shape and (Kd != 0).nnz >= (Ko != 0).nnz
            assert abs(Kd - Ko).max() <= 1e-13 * abs(Ko).max(), l
            rows.append(int(np.diff(Kd.indptr).max()) // 2)
        for l in range(1, levels + 1):
            Pd, Po = b.level_transfer(l), mg.P[l]
            assert Pd.shape == Po.shape
            assert abs(Pd - Po).max() <= 1e-14, l
            a, o = Pd.copy(), Po.copy()
            a.data[:], o.data[:] = 1.0, 1.0
            assert (a != o).nnz == 0, l
    print("%s: level vertices %s, most blocks per row %s" % (name, [x["n_vertices"] for x in lv], rows))
    assert max(rows) <= 63


def test_two_builds_and_solves_give_the_same_bits(ctx):
    s, _ = jittered_case("cantilever", 3)
    out = []
    for _ in range(2):
        with ctx.create_batch(pack([s])) as b:
            b.set_grid_hierarchy(4).assemble()
            K0 = b.level_csr(0)
            r = b.solve(RTOL, MAX_ITER).download()
        out.append((K0, r))
    (ka, ra), (kb, rb) = out
    assert ka.data.tobytes() == kb.data.tobytes() and np.array_equal(ka.indices, kb.indices)
    assert ra.u.tobytes() == rb.u.tobytes() and np.array_equal(ra.iters, rb.iters) and ra.relres.tobytes() == rb.relres.tobytes()


def _against_block_jacobi(ctx, packed, levels, tag):
    with ctx.create_batch(packed) as b:
        r = b.set_grid_hierarchy(levels).assemble().solve(RTOL, MAX_ITER).download()
        st = b.stats()
    with ctx.create_batch(packed) as b:
        ref = b.assemble().solve(RTOL, 400000).download()
    print("%s: grid hierarchy %d outer iterations, block-Jacobi CG %d iterations, rel-L2 %.2e" % (
        tag, st["iterations"], ref.iters[0], rel(r.u, ref.u)))
    assert r.status[0] == SAMPLE_CONVERGED and ref.status[0] == SAMPLE_CONVERGED
    assert rel(r.u, ref.u) <= 1e-9
    return r


def test_jittered_cantilever_l3_converges(ctx):
    s, _ = jittered_case("cantilever", 3)
    _against_block_jacobi(ctx, pack([s]), 4, "jittered cantilever-L3")


def test_plate_from_description_and_from_conditions(ctx):
    s, (coors, conn), kw = plate(0.0025)
    a = _against_block_jacobi(ctx, pack([s]), 4, "plate h=0.0025")
    b = _against_block_jacobi(ctx, PackedConditions([(coors, conn)], [(0, kw)]), 4, "plate h=0.0025 from conditions")
    assert rel(a.u, b.u) <= 1e-9


def test_cantilever_l4_matches_the_stored_sparse_lu_solution(ctx):
    """Solved through the grid hierarchy without declaring its refinement."""
    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "c3_lu.npz"))
    setup, n0 = large_case("cantilever", 4)
    with ctx.create_batch(pack([setup.sample])) as b:
        r = b.set_grid_hierarchy(5).assemble().solve(RTOL, MAX_ITER).download()
    g = ref["cantilever_L4_u_coarse"]
    assert r.status[0] == SAMPLE_CONVERGED
    assert rel(r.u[:n0], g) <= 1e-8


@pytest.mark.parametrize("K", [3, 8])
def test_load_cases_are_bitwise_their_single_solves(ctx, K):
    s, _ = jittered_case("cantilever", 2)
    free = ~s.fixed.astype(bool)
    rng = np.random.default_rng(K)
    loads = np.zeros((K,) + s.rhs.shape)
    loads[0] = s.rhs
    for k in range(1, K):
        loads[k][free] = rng.uniform(-100.0, 100.0, (int(free.sum()), 2))
    loads[K - 1][np.flatnonzero(free)[0]] = (np.nan, 0.0)
    lo, hi = s.coors.min(0), s.coors.max(0)
    size = 97
    scale = (size - 1) / (hi - lo).max()
    aff = np.array([scale, -scale * lo[0], scale, -scale * lo[1]])
    with ctx.create_batch(pack([s])) as b:
        res = b.set_grid_hierarchy(3).assemble().solve_load_cases(loads, RTOL, MAX_ITER)
        images = b.load_case_images(size, aff)
    assert images.shape == (K, 2, size, size)
    assert res.status[K - 1] == SAMPLE_BREAKDOWN and (res.status[:K - 1] == SAMPLE_CONVERGED).all()
    for k in range(K):
        with ctx.create_batch(pack([with_rhs(s, loads[k])])) as b:
            r = b.set_grid_hierarchy(3).assemble().solve(RTOL, MAX_ITER).rasterize(size, aff[None], 1.0).download(images=True)
        for x, y in ((res.u[k], r.u), (res.ranges[k], r.ranges[0]), (res.iters[k], r.iters[0]),
                     (res.relres[k], r.relres[0]), (res.status[k], r.status[0]), (images[k], r.images[0])):
            assert np.asarray(x).tobytes() == np.asarray(y).tobytes(), k


def _code(fn):
    try:
        fn()
    except FeaError as e:
        return e.code
    return 0


def test_return_codes(ctx):
    s = plate(0.02)[0]
    lib = ctx.lib

    def with_batch(samples, act):
        with ctx.create_batch(pack(samples)) as b:
            return _code(lambda: act(b))

    # BAD_ARG: two samples, quads, levels outside 1..8
    assert with_batch([s, s], lambda b: b.set_grid_hierarchy(2)) == BAD_ARG
    xy = np.array([[0, 0], [1, 0], [2, 0], [0, 1], [1, 1], [2, 1]], np.float64)
    q = Sample(xy, np.array([[0, 1, 4, 3], [1, 2, 5, 4]], np.int32), np.zeros(2, np.int8), s.D[:1],
               np.array([1, 0, 0, 1, 0, 0], np.uint8), np.zeros((6, 2)))
    assert with_batch([q], lambda b: b.set_grid_hierarchy(1)) == BAD_ARG
    for levels in (0, 9, -1):
        assert with_batch([s], lambda b: ctx._check(lib.fea_batch_set_grid_hierarchy(b.h, levels))) == BAD_ARG
    assert lib.fea_batch_set_grid_hierarchy(None, 2) == BAD_ARG
    # BAD_STATE: after assemble, after any hierarchy
    assert with_batch([s], lambda b: b.assemble().set_grid_hierarchy(2)) == BAD_STATE
    assert with_batch([s], lambda b: b.set_grid_hierarchy(2).set_grid_hierarchy(2)) == BAD_STATE
    coarse = pack([ProblemSetup(*plate_meshes(1, [0.04])[0][0], **plate(0.02)[2]).sample])
    assert with_batch([s], lambda b: b.set_coarse_meshes(coarse).set_grid_hierarchy(2)) == BAD_STATE
    assert with_batch([s], lambda b: b.set_grid_hierarchy(2).set_coarse_meshes(coarse)) == BAD_STATE
    s1 = large_case("cantilever", 1)[0].sample
    assert with_batch([s1], lambda b: b.set_refinement(1).set_grid_hierarchy(1)) == BAD_STATE
    assert with_batch([s1], lambda b: b.set_grid_hierarchy(1).set_refinement(1)) == BAD_STATE
    # a build that fails (no active vertex to lay grids under) leaves the batch unassembled for good
    fixed = Sample(s.coors, s.conn, s.cell_region, s.D, np.ones_like(s.fixed), s.rhs)
    with ctx.create_batch(pack([fixed])) as b:
        b.set_grid_hierarchy(2)
        assert _code(b.assemble) == MESH_ERROR
        assert _code(lambda: b.solve(RTOL, MAX_ITER)) == BAD_STATE
        assert _code(b.assemble) == BAD_STATE
    # the levels and load cases need an assembled batch
    with ctx.create_batch(pack([s])) as b:
        b.set_grid_hierarchy(2)
        assert _code(lambda: b.mg_levels()) == BAD_STATE
        assert _code(lambda: b.solve_load_cases(s.rhs[None].copy())) == BAD_STATE
        r = b.assemble().solve(RTOL, MAX_ITER).download()
        assert r.status[0] == SAMPLE_CONVERGED
