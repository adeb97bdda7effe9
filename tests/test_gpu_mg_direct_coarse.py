"""Direct coarsest-level solver of the multigrid V-cycle (fea_batch_set_coarse_solver(b, FEA_COARSE_DIRECT)): the coarse
solve against a sparse direct solve for every hierarchy kind, the V-cycle as a symmetric positive operator, solves,
determinism, load cases bit for bit against single solves, and the return codes."""
import ctypes as C
import os

import numpy as np
import pytest

import cases
from fea_diffusion_b200 import Context, FeaError, pack
from fea_diffusion_b200._capi import SAMPLE_BREAKDOWN, SAMPLE_CONVERGED, CoarseInfo
from fea_diffusion_b200.host import ProblemSetup
from fea_diffusion_b200.solver import Sample
from fea_diffusion_b200.workload import jittered_case, large_case, plate_condition, plate_meshes
from oracle.multigrid import Multigrid

pytestmark = pytest.mark.gpu

BAD_ARG, BAD_STATE, MESH_ERROR = 1, 4, 5
RTOL, MAX_ITER = 1e-10, 200


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


def with_rhs(s, rhs):
    return Sample(s.coors, s.conn, s.cell_region, s.D, s.fixed, np.ascontiguousarray(rhs))


def refined(level):
    return large_case("cantilever", level)[0].sample, lambda b: b.set_refinement(level)


def jittered(level):
    s, _ = jittered_case("cantilever", level)
    coarse = pack([large_case("cantilever", l)[0].sample for l in range(level)])
    return s, lambda b: b.set_coarse_meshes(coarse)


def grid_plate():
    (mesh,), ptags, ltags = plate_meshes(1, [0.005])
    s = ProblemSetup(mesh[0], mesh[1], **plate_condition(ptags, ltags)).sample
    return s, lambda b: b.set_grid_hierarchy(2)


HIERARCHIES = {"refinement-cantilever-L2": lambda: refined(2), "coarse-meshes-jittered-L3": lambda: jittered(3),
               "grid-plate-0.005": grid_plate}


def _code(fn):
    try:
        fn()
    except FeaError as e:
        return e.code
    return 0


def assembled(ctx, s, declare, solver):
    b = ctx.create_batch(pack([s]))
    declare(b)
    if solver is not None:
        b.set_coarse_solver(solver)
    return b.assemble()


@pytest.mark.parametrize("name", sorted(HIERARCHIES))
def test_coarse_solve_matches_a_sparse_direct_solve(ctx, name):
    import scipy.sparse.linalg as spla
    s, declare = HIERARCHIES[name]()
    with assembled(ctx, s, declare, "direct") as b:
        K0 = b.level_csr(0)
        r = np.random.default_rng(3).standard_normal(K0.shape[0])
        x = b.coarse_solve(r)
        info = b.coarse_info()
    ref = spla.spsolve(K0.tocsc(), r)
    err = float(np.linalg.norm(x - ref) / np.linalg.norm(ref))
    print("%s: level-0 DOFs %d, coarse solve rel-L2 %.3e, smallest pivot %.4e, factor %.2f ms" %
          (name, K0.shape[0], err, info["min_pivot"], info["n"] and info["factor_ms"]))
    assert info["solver"] == 1 and info["n"] == K0.shape[0]
    assert info["bytes"] >= 8 * K0.shape[0] ** 2 and 0.0 < info["min_pivot"] <= 1.0
    assert err <= 1e-8


def test_cg_coarse_solve_is_the_vcycle_s_inexact_one(ctx):
    from oracle.multigrid import block_scaling
    s, declare = refined(2)
    with assembled(ctx, s, declare, None) as b:
        K0 = b.level_csr(0)
        r = np.random.default_rng(3).standard_normal(K0.shape[0])
        x = b.coarse_solve(r)
        assert b.coarse_info() == {"solver": 0, "n": 0, "factor_ms": 0.0, "min_pivot": 0.0, "bytes": 0}
    S = block_scaling(K0)
    rel = float(np.linalg.norm(S.T @ (r - K0 @ x)) / np.linalg.norm(S.T @ r))
    print("CG coarse solve: scaled relative residual %.3e" % rel)
    assert 0.0 < rel <= 1.5e-4


def test_vcycle_is_symmetric_positive_and_contracts(ctx):
    s, declare = refined(2)
    mg = Multigrid(s.coors, s.conn, s.cell_region, s.D, s.fixed, 2)
    with assembled(ctx, s, declare, "direct") as b:
        K = b.csr(0)
        rng = np.random.default_rng(11)
        a, c = rng.standard_normal(K.shape[0]), rng.standard_normal(K.shape[0])
        Ma, Mc = b.mg_apply(a), b.mg_apply(c)
        x = rng.standard_normal(K.shape[0])
        e = x - b.mg_apply(K @ x)
    asym = abs(a @ Mc - c @ Ma)
    assert asym <= 1e-10 * np.linalg.norm(a) * np.linalg.norm(Mc), asym
    assert a @ Ma > 0 and c @ Mc > 0
    ratio = np.sqrt(e @ (K @ e)) / np.sqrt(x @ (K @ x))
    eo = x - mg.apply_unscaled(K @ x)
    ref = np.sqrt(eo @ (K @ eo)) / np.sqrt(x @ (K @ x))
    print("V-cycle with the direct coarse solve: energy contraction %.4f (numpy, exact coarse solve: %.4f), "
          "asymmetry %.2e" % (ratio, ref, asym / (np.linalg.norm(a) * np.linalg.norm(Mc))))
    assert ratio <= 0.3 and abs(ratio - ref) <= 0.02


def test_cantilever_l4_matches_the_stored_sparse_lu_solution(ctx):
    ref = np.load(os.path.join(cases.ROOT, "tests", "golden", "c3_lu.npz"))
    setup, n0 = large_case("cantilever", 4)
    with assembled(ctx, setup.sample, lambda b: b.set_refinement(4), "direct") as b:
        r = b.solve(RTOL, MAX_ITER).download()
        st, info = b.stats(), b.coarse_info()
    g = ref["cantilever_L4_u_coarse"]
    err = float(np.linalg.norm(r.u[:n0] - g) / np.linalg.norm(g))
    print("cantilever-L4: %d outer iterations, %.2f ms, rel-L2 %.3e vs LU, factor %.2f ms of n = %d" %
          (st["iterations"], st["solve_ms"], err, info["factor_ms"], info["n"]))
    assert r.status[0] == SAMPLE_CONVERGED and err <= 1e-8


@pytest.mark.parametrize("name", ["refinement-cantilever-L3", "coarse-meshes-jittered-L3", "grid-plate-0.005"])
def test_direct_takes_no_more_outer_iterations_than_cg(ctx, name):
    s, declare = refined(3) if name == "refinement-cantilever-L3" else HIERARCHIES[name]()
    its, us = {}, {}
    for solver in ("cg", "direct"):
        with assembled(ctx, s, declare, solver) as b:
            r = b.solve(RTOL, MAX_ITER).download()
            assert r.status[0] == SAMPLE_CONVERGED
            its[solver], us[solver] = int(r.iters[0]), r.u
    print("%s: outer iterations cg %d, direct %d" % (name, its["cg"], its["direct"]))
    assert its["direct"] <= its["cg"] + 1
    assert np.linalg.norm(us["direct"] - us["cg"]) <= 1e-8 * np.linalg.norm(us["cg"])


def test_two_builds_give_the_same_bits_and_cg_is_the_default(ctx):
    s, declare = jittered(3)
    out = []
    for solver in ("direct", "direct", "cg", None):
        with assembled(ctx, s, declare, solver) as b:
            r = b.solve(RTOL, MAX_ITER).download()
            out.append((r.u.tobytes(), r.relres.tobytes(), r.iters.tobytes(), r.status.tobytes(),
                        b.coarse_info()["min_pivot"]))
    assert out[0] == out[1]
    assert out[2] == out[3]
    assert out[0][0] != out[2][0]


def single(ctx, s, declare, rhs):
    with assembled(ctx, with_rhs(s, rhs), declare, "direct") as b:
        r = b.solve(RTOL, MAX_ITER).download()
    return r.u, r.ranges[0], r.iters[0], r.relres[0], r.status[0]


@pytest.mark.parametrize("name", ["refinement-cantilever-L2", "coarse-meshes-jittered-L3"])
def test_load_cases_are_bitwise_their_single_direct_solves(ctx, name):
    s, declare = HIERARCHIES[name]()
    free = np.flatnonzero(~s.fixed.astype(bool))
    point = np.zeros_like(s.rhs)
    point[free[np.argmax(s.coors[free, 0])]] = (1000.0, 0.0)
    rnd = np.zeros_like(s.rhs)
    rnd[free] = np.random.default_rng(7).uniform(-100.0, 100.0, (len(free), 2))
    nan = s.rhs.copy()
    nan[free[5]] = (np.nan, 0.0)
    loads = [s.rhs, point, rnd, nan, np.zeros_like(s.rhs)]
    ref = [single(ctx, s, declare, f) for f in loads]
    assert ref[3][4] == SAMPLE_BREAKDOWN
    with assembled(ctx, s, declare, "direct") as b:
        for order in ([0, 3, 1], [2, 0, 3, 1, 0, 4, 2, 1]):
            res = b.solve_load_cases(np.stack([loads[k] for k in order]), RTOL, MAX_ITER)
            for i, k in enumerate(order):
                got = (res.u[i], res.ranges[i], res.iters[i], res.relres[i], res.status[i])
                assert all(np.asarray(x).tobytes() == np.asarray(y).tobytes() for x, y in zip(got, ref[k])), (order, i)
            print(name, "K = %d: outer iterations" % len(order), res.iters.tolist(), "status", res.status.tolist(),
                  "solve ms %.2f" % res.stats["solve_ms"])


def test_return_codes(ctx):
    lib = ctx.lib
    s, declare = refined(1)
    info = CoarseInfo()
    x = np.zeros(4)
    with ctx.create_batch(pack([s])) as b:   # no hierarchy
        assert _code(lambda: b.set_coarse_solver("direct")) == BAD_STATE
        assert lib.fea_batch_get_coarse_info(b.h, C.byref(info)) == BAD_STATE
        assert lib.fea_batch_coarse_solve(b.h, x.ctypes.data_as(C.c_void_p), x.ctypes.data_as(C.c_void_p)) == BAD_STATE
    with ctx.create_batch(pack([s])) as b:
        declare(b)
        for solver in (2, -1):
            assert lib.fea_batch_set_coarse_solver(b.h, solver) == BAD_ARG
        assert lib.fea_batch_get_coarse_info(b.h, C.byref(info)) == BAD_STATE           # before assemble
        assert lib.fea_batch_coarse_solve(b.h, x.ctypes.data_as(C.c_void_p), x.ctypes.data_as(C.c_void_p)) == BAD_STATE
        b.set_coarse_solver("cg").set_coarse_solver("direct")                           # the last call counts
        b.assemble()
        assert b.coarse_info()["solver"] == 1
        assert _code(lambda: b.set_coarse_solver("cg")) == BAD_STATE                   # after assemble
        assert lib.fea_batch_coarse_solve(b.h, None, x.ctypes.data_as(C.c_void_p)) == BAD_ARG
        assert lib.fea_batch_coarse_solve(b.h, x.ctypes.data_as(C.c_void_p), None) == BAD_ARG
        assert lib.fea_batch_get_coarse_info(b.h, None) == BAD_ARG
    # gusset-L1 refined once: level 0 has 19 996 DOFs, over the 16 384 of the dense inverse
    g = large_case("gusset", 1)[0].sample
    with ctx.create_batch(pack([g])) as b:
        b.set_refinement(1).set_coarse_solver("direct")
        with pytest.raises(FeaError) as e:
            b.assemble()
        print("gusset-L1:", e.value)
        assert e.value.code == MESH_ERROR and "19996" in str(e.value)
        assert _code(b.assemble) == BAD_STATE
        assert _code(lambda: b.solve(RTOL, MAX_ITER)) == BAD_STATE
    # a floating coarsest mesh (no fixed vertex): Khat_0 is singular, a pivot falls to rounding level
    s3, _ = jittered(2)
    coarse = [large_case("cantilever", l)[0].sample for l in range(2)]
    coarse[0] = Sample(coarse[0].coors, coarse[0].conn, coarse[0].cell_region, coarse[0].D,
                       np.zeros_like(coarse[0].fixed), coarse[0].rhs)
    with ctx.create_batch(pack([s3])) as b:
        b.set_coarse_meshes(pack(coarse)).set_coarse_solver("direct")
        with pytest.raises(FeaError) as e:
            b.assemble()
        print("floating level 0:", e.value)
        assert e.value.code == MESH_ERROR and "pivot" in str(e.value)
        assert _code(b.assemble) == BAD_STATE
    # the smallest pivots of legitimate levels 0, for the threshold between them and the floating one
    for name in sorted(HIERARCHIES):
        sh, dh = HIERARCHIES[name]()
        with assembled(ctx, sh, dh, "direct") as b:
            print("%s: smallest pivot %.4e" % (name, b.coarse_info()["min_pivot"]))
