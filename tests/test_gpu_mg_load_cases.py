"""Several load cases of one multigrid batch in one call (fea_batch_solve_load_cases): every case bit for bit
the single solve of a batch created with that load, whatever cases share the call; accuracy against a direct
solve and superposition; the batch's own state; return codes."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest
import scipy.sparse.linalg as spla

from fea_diffusion_b200 import Context, FeaError, pack
from fea_diffusion_b200.host import MeshTopology, ProblemSetup, vertices_on_line
from fea_diffusion_b200.solver import Sample
from fea_diffusion_b200._capi import SAMPLE_BREAKDOWN, SAMPLE_CONVERGED, SolveStats, ptr
from fea_diffusion_b200.workload import jittered_case, large_case, plate_condition, plate_meshes

pytestmark = pytest.mark.gpu

BAD_ARG, BAD_STATE = 1, 4
RTOL, MAX_ITER = 1e-10, 200


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


def with_rhs(s, rhs):
    return Sample(s.coors, s.conn, s.cell_region, s.D, s.fixed, np.ascontiguousarray(rhs))


def cantilever_refined(level):
    s = large_case("cantilever", level)[0].sample
    return s, lambda b: b.set_refinement(level)


def cantilever_jittered(level):
    s, _ = jittered_case("cantilever", level)
    coarse = pack([large_case("cantilever", l)[0].sample for l in range(level)])
    return s, lambda b: b.set_coarse_meshes(coarse)


def plate(sizes):
    meshes, ptags, ltags = plate_meshes(1, sizes)
    kw = plate_condition(ptags, ltags)
    levels = [ProblemSetup(c, n, **kw).sample for c, n in meshes]
    coarse = pack(levels[:-1])
    return levels[-1], lambda b: b.set_coarse_meshes(coarse)


MESHES = {
    "cantilever-L3-refinement": lambda: cantilever_refined(3),
    "plate-0.01-coarse-meshes": lambda: plate([0.04, 0.02, 0.01]),
    "cantilever-L3-jittered-coarse-meshes": lambda: cantilever_jittered(3),
}


def five_loads(s):
    """The model's own load, a horizontal point load, a load on the right edge, a seeded random load on every
    free vertex, and zero."""
    free = ~s.fixed.astype(bool)
    x = s.coors[:, 0]
    point = np.zeros_like(s.rhs)
    point[np.flatnonzero(free)[np.argmax(x[free])]] = (1000.0, 0.0)
    edge = np.zeros_like(s.rhs)
    edge[free & (x >= x.max() - 1e-9 * (x.max() - x.min()))] = (0.0, -250.0)
    rnd = np.zeros_like(s.rhs)
    rnd[free] = np.random.default_rng(7).uniform(-100.0, 100.0, (int(free.sum()), 2))
    return np.stack([s.rhs, point, edge, rnd, np.zeros_like(s.rhs)])


def single(ctx, s, declare, rhs):
    with ctx.create_batch(pack([with_rhs(s, rhs)])) as b:
        declare(b)
        r = b.assemble().solve(RTOL, MAX_ITER).download()
    return r.u, r.ranges[0], r.iters[0], r.relres[0], r.status[0]


def case(res, k):
    return res.u[k], res.ranges[k], res.iters[k], res.relres[k], res.status[k]


def same_bytes(a, b):
    return all(np.asarray(x).tobytes() == np.asarray(y).tobytes() for x, y in zip(a, b))


@pytest.fixture(scope="module", params=sorted(MESHES))
def mesh(request, ctx):
    s, declare = MESHES[request.param]()
    loads = five_loads(s)
    b = ctx.create_batch(pack([s]))
    declare(b)
    b.assemble()
    ref = [single(ctx, s, declare, loads[k]) for k in range(len(loads))]
    yield request.param, s, loads, b, ref
    b.destroy()


def test_every_case_is_bitwise_its_single_solve(mesh):
    name, s, loads, b, ref = mesh
    res = b.solve_load_cases(loads, RTOL, MAX_ITER)
    print(name, "outer iterations per case", res.iters.tolist(), "status", res.status.tolist(),
          "solve ms", round(res.stats["solve_ms"], 2))
    assert res.u.shape == (5, len(s.coors), 2) and res.ranges.shape == (5, 4)
    for k in range(5):
        assert same_bytes(case(res, k), ref[k]), "case %d" % k
    assert res.stats["iterations"] == res.iters.max()
    assert res.stats["n_converged"] == int((res.status == SAMPLE_CONVERGED).sum())


def test_cases_do_not_depend_on_their_company(mesh):
    name, s, loads, b, ref = mesh
    for order in ([4, 3, 2, 1, 0], [1, 3], [0, 2, 4], [3, 0, 1, 2, 4, 3, 0, 1], [2, 4, 1, 0, 3, 1], [0, 1, 2, 3, 4, 2, 0]):
        res = b.solve_load_cases(loads[order], RTOL, MAX_ITER)
        for i, k in enumerate(order):
            assert same_bytes(case(res, i), ref[k]), (order, i)
    for k in range(5):
        assert same_bytes(case(b.solve_load_cases(loads[k:k + 1], RTOL, MAX_ITER), 0), ref[k])


def test_a_nan_load_breaks_down_alone(mesh):
    name, s, loads, b, ref = mesh
    bad = loads[3].copy()
    bad[np.flatnonzero(~s.fixed.astype(bool))[5]] = (np.nan, 0.0)
    res = b.solve_load_cases(np.stack([loads[0], bad, loads[3], loads[2]]), RTOL, MAX_ITER)
    assert res.status[1] == SAMPLE_BREAKDOWN
    for i, k in ((0, 0), (2, 3), (3, 2)):
        assert same_bytes(case(res, i), ref[k]), i


def test_single_solves_keep_the_bits_of_the_solver_before_load_cases(ctx):
    """fea_batch_solve on a multigrid batch runs the one-case instance of the load-case driver; its outputs are
    those of the solver before load cases existed (digests of that build's outputs on a B200)."""
    with open(os.path.join(os.path.dirname(__file__), "golden", "mg_solve_digests.json")) as f:
        want = json.load(f)["meshes"]
    jc = pack([large_case("cantilever", l)[0].sample for l in range(3)])
    runs = {"cantilever-L3": (large_case("cantilever", 3)[0].sample, lambda b: b.set_refinement(3)),
            "gusset-L2": (large_case("gusset", 2)[0].sample, lambda b: b.set_refinement(2)),
            "jittered-cantilever-L3": (jittered_case("cantilever", 3)[0], lambda b: b.set_coarse_meshes(jc))}
    for name, (s, declare) in runs.items():
        with ctx.create_batch(pack([s])) as b:
            declare(b)
            r = b.assemble().solve(1e-10, 400000).download()
        got = {f + "_sha256": hashlib.sha256(np.ascontiguousarray(getattr(r, f)).tobytes()).hexdigest()
               for f in ("u", "ranges", "iters", "relres", "status")}
        assert int(r.iters[0]) == want[name]["iters"] and int(r.status[0]) == want[name]["status"], name
        assert got == {k: v for k, v in want[name].items() if k.endswith("_sha256")}, name


def test_cases_match_a_direct_solve(ctx):
    s, declare = cantilever_refined(2)
    loads = five_loads(s)
    act = ~s.fixed.astype(bool)
    with ctx.create_batch(pack([s])) as b:
        declare(b)
        res = b.assemble().solve_load_cases(loads, RTOL, MAX_ITER)
        lu = spla.splu(b.csr(0).tocsc())
    for k in range(4):
        u = np.zeros_like(s.rhs)
        u[act] = lu.solve(loads[k][act].reshape(-1)).reshape(-1, 2)
        assert np.linalg.norm(res.u[k] - u) <= 1e-8 * np.linalg.norm(u), k
    assert not res.u[4].any()


def test_gusset_loads_superpose(ctx):
    setup, _ = large_case("gusset", 2)
    s = setup.sample
    co = s.coors
    topo = MeshTopology(setup.conn, len(co))
    edge, line = np.zeros_like(s.rhs), np.zeros_like(s.rhs)
    edge[topo.facet_vertices(np.flatnonzero(co[:, 0] > 0.99))] += (1000.0, 0.0)
    line[topo.facet_vertices(vertices_on_line(co, (3, 4)))] += (1000.0, 1000.0)
    with ctx.create_batch(pack([s])) as b:
        res = b.set_refinement(2).assemble().solve_load_cases(np.stack([edge, line, edge + line]), RTOL, MAX_ITER)
    assert (res.status == SAMPLE_CONVERGED).all()
    both = res.u[2]
    assert np.linalg.norm(res.u[0] + res.u[1] - both) <= 1e-9 * np.linalg.norm(both)
    assert np.array_equal(edge + line, s.rhs)   # the model's own load is the sum of the two


def test_the_batch_keeps_its_own_results(ctx):
    s, declare = cantilever_refined(3)
    loads = five_loads(s)
    with ctx.create_batch(pack([s])) as fresh:
        declare(fresh)
        want = fresh.assemble().solve(RTOL, MAX_ITER).download()
    with ctx.create_batch(pack([s])) as b:
        declare(b)
        before = b.assemble().solve(RTOL, MAX_ITER).download()
        res = b.solve_load_cases(loads[[3, 1]], RTOL, MAX_ITER)
        lv = b.mg_levels()
        after = b.download()
        again = b.solve(RTOL, MAX_ITER).download()
    for r in (before, after, again):
        assert same_bytes((r.u, r.ranges, r.iters, r.relres, r.status), (want.u, want.ranges, want.iters, want.relres, want.status))
    assert all(x["vcycle_ms"] > 0.0 for x in lv)
    assert res.stats["iterations"] == res.iters.max()
    with ctx.create_batch(pack([s])) as b:
        declare(b)
        z = b.assemble().solve_load_cases(np.zeros((1, len(s.coors), 2)), RTOL, MAX_ITER)
    assert z.status[0] == SAMPLE_CONVERGED and z.iters[0] == 0 and not z.u.any()


def test_return_codes(ctx):
    s, declare = cantilever_refined(1)
    lib = ctx.lib
    nv = len(s.coors)
    loads = np.zeros((9, nv, 2))

    def raw(b, n, rhs, rtol=RTOL, max_iter=MAX_ITER):
        st = SolveStats()
        return lib.fea_batch_solve_load_cases(b.h, n, ptr(rhs) if rhs is not None else None, rtol, max_iter,
                                              None, None, None, None, None, C.byref(st))

    with ctx.create_batch(pack([s])) as b:           # no hierarchy
        assert raw(b.assemble(), 1, loads) == BAD_STATE
    with ctx.create_batch(pack([s])) as b:           # not assembled
        declare(b)
        assert raw(b, 1, loads) == BAD_STATE
        b.assemble()
        assert raw(b, 0, loads) == BAD_ARG
        assert raw(b, 9, loads) == BAD_ARG
        assert raw(b, 1, None) == BAD_ARG
        assert raw(b, 1, loads, rtol=-1.0) == BAD_ARG
        assert raw(b, 1, loads, max_iter=0) == BAD_ARG
        with pytest.raises(FeaError) as e:
            b.solve_load_cases(loads)
        assert e.value.code == BAD_ARG
        assert raw(b, 8, loads) == 0                  # outputs may all be NULL
