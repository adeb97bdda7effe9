"""Outputs of every load case of a multigrid call from the displacements kept on the device
(fea_batch_load_case_images / _strain_stress / _cell_components): each case bit for bit what the single-batch
outputs give a batch created with that load, for both hierarchy kinds; the state rules and return codes."""
import numpy as np
import pytest

from fea_diffusion_b200 import Context, FeaError, pack
from fea_diffusion_b200._capi import SAMPLE_BREAKDOWN, ptr
from fea_diffusion_b200.imaging import crop_affine, plate_window
from fea_diffusion_b200.solver import Sample
from fea_diffusion_b200.workload import jittered_case, large_case

pytestmark = pytest.mark.gpu

BAD_ARG, BAD_STATE = 1, 4
RTOL, MAX_ITER = 1e-10, 200
SIZE, SCALE = 97, 0.37   # 97^2 pixels: the last 256-thread block of the shading kernels is partial
NAMES = ["stress_x", "stress_y", "strain_x", "strain_y"]


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


def refined(level):
    return large_case("cantilever", level)[0].sample, lambda b: b.set_refinement(level)


def jittered(level):
    s, _ = jittered_case("cantilever", level)
    coarse = pack([large_case("cantilever", l)[0].sample for l in range(level)])
    return s, lambda b: b.set_coarse_meshes(coarse)


MESHES = {"cantilever-L2-refinement": lambda: refined(2), "cantilever-L3-jittered-coarse-meshes": lambda: jittered(3)}


def camera(s):
    x, y = s.coors[:, 0], s.coors[:, 1]
    bbox = (x.min(), y.min(), x.max(), y.max())
    window, bounds = plate_window(bbox, SIZE)
    return crop_affine(bbox, window, bounds)


def six_loads(s):
    """The model's own load, a point load, a right-edge load, a seeded random load, zero, and a NaN load."""
    free = np.flatnonzero(~s.fixed.astype(bool))
    x = s.coors[:, 0]
    point = np.zeros_like(s.rhs)
    point[free[np.argmax(x[free])]] = (1000.0, 0.0)
    edge = np.zeros_like(s.rhs)
    edge[free[x[free] >= x.max() - 1e-9 * (x.max() - x.min())]] = (0.0, -250.0)
    rnd = np.zeros_like(s.rhs)
    rnd[free] = np.random.default_rng(7).uniform(-100.0, 100.0, (len(free), 2))
    nan = rnd.copy()
    nan[free[5]] = (np.nan, 0.0)
    return np.ascontiguousarray(np.stack([s.rhs, point, edge, rnd, np.zeros_like(s.rhs), nan]))


def outputs_of_single(ctx, s, declare, rhs, affine):
    """What the single-batch outputs give a batch created with load rhs."""
    with ctx.create_batch(pack([Sample(s.coors, s.conn, s.cell_region, s.D, s.fixed, np.ascontiguousarray(rhs))])) as b:
        declare(b)
        r = b.assemble().solve(RTOL, MAX_ITER).rasterize(SIZE, affine.reshape(1, 4), SCALE).download(images=True)
        out = {"status": int(r.status[0]), "images": r.images[0]}
        for region in (-1, 0):
            out["strain", region], out["stress", region] = b.cell_strain_stress(region)
            out["components", region] = b.rasterize_cell_components(region, NAMES, SCALE)
    return out


def outputs_of_cases(b, affine):
    out = {"images": b.load_case_images(SIZE, affine, SCALE)}
    for region in (-1, 0):
        out["strain", region], out["stress", region] = b.load_case_strain_stress(region)
        out["components", region] = b.load_case_cell_components(region, NAMES, SCALE)
    return out


def same_floats(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def assert_case_is_single(got, k, want, what):
    assert np.array_equal(got["images"][k], want["images"]), what
    for region in (-1, 0):
        assert same_floats(got["strain", region][k], want["strain", region]), (what, "strain", region)
        assert same_floats(got["stress", region][k], want["stress", region]), (what, "stress", region)
        imgs, rngs = got["components", region]
        want_imgs, want_rngs = want["components", region]
        for nm in NAMES:
            assert np.array_equal(imgs[nm][k], want_imgs[nm][0]), (what, nm, region)
            assert same_floats(rngs[nm][k], want_rngs[nm][0]), (what, nm, region, "range")


@pytest.fixture(scope="module", params=sorted(MESHES))
def mesh(request, ctx):
    s, declare = MESHES[request.param]()
    loads = six_loads(s)
    affine = camera(s)
    ref = [outputs_of_single(ctx, s, declare, loads[k], affine) for k in range(len(loads))]
    assert ref[5]["status"] == SAMPLE_BREAKDOWN
    b = ctx.create_batch(pack([s]))
    declare(b)
    b.assemble()
    yield request.param, s, loads, affine, b, ref
    b.destroy()


@pytest.mark.parametrize("order", [[5, 2, 0], [3, 0, 5, 2, 1, 0, 4, 3]], ids=["K3", "K8"])
def test_every_case_is_bitwise_its_single_batch(mesh, order):
    name, s, loads, affine, b, ref = mesh
    res = b.solve_load_cases(loads[order], RTOL, MAX_ITER)
    assert res.status[order.index(5)] == SAMPLE_BREAKDOWN
    got = outputs_of_cases(b, affine)
    K, nc = len(order), len(s.conn)
    assert got["images"].shape == (K, 2, SIZE, SIZE)
    assert got["strain", -1].shape == got["stress", 0].shape == (K, nc, 3)
    assert got["components", 0][0]["stress_x"].shape == (K, SIZE, SIZE)
    assert got["components", 0][1]["strain_y"].shape == (K, 2)
    for i, k in enumerate(order):
        assert_case_is_single(got, i, ref[k], (name, order, i))


def test_state_rules(ctx):
    s, declare = refined(2)
    loads = six_loads(s)
    affine = camera(s)
    lib = ctx.lib
    nc = len(s.conn)
    img = np.empty((8, 2, SIZE, SIZE), np.uint8)
    strain = np.empty((8, nc, 3))
    ids = np.arange(4, dtype=np.int32)
    rng = np.empty((4, 8, 2))
    cimg = np.empty((4, 8, SIZE, SIZE), np.uint8)

    def raw_images(b, size=SIZE, aff=affine, out=img):
        return lib.fea_batch_load_case_images(b.h, size, ptr(aff) if aff is not None else None, SCALE,
                                              ptr(out) if out is not None else None)

    def raw_strain(b):
        return lib.fea_batch_load_case_strain_stress(b.h, -1, ptr(strain), None)

    def raw_components(b, n=4, field_ids=ids):
        return lib.fea_batch_load_case_cell_components(b.h, 0, n, ptr(field_ids), SCALE, ptr(cimg), ptr(rng))

    with ctx.create_batch(pack([s])) as b:           # no hierarchy: no load-case call can have succeeded
        b.assemble().solve(RTOL, MAX_ITER)
        assert raw_images(b) == raw_strain(b) == raw_components(b) == BAD_STATE
    with ctx.create_batch(pack([s])) as b:
        declare(b)
        b.assemble().solve(RTOL, MAX_ITER).rasterize(SIZE, affine.reshape(1, 4), SCALE)
        own = b.download(images=True)
        own_components = b.rasterize_cell_components(-1, NAMES, SCALE)
        assert raw_images(b) == raw_strain(b) == raw_components(b) == BAD_STATE
        for call in (b.load_case_info, lambda: b.load_case_images(SIZE, affine), b.load_case_strain_stress,
                     lambda: b.load_case_cell_components(0, NAMES)):
            with pytest.raises(FeaError) as e:
                call()
            assert e.value.code == BAD_STATE

        b.solve_load_cases(loads[[0, 1, 2, 3, 4, 0, 1, 2]], RTOL, MAX_ITER)
        assert raw_components(b) == BAD_STATE             # needs the camera of a load_case_images call
        with pytest.raises(FeaError) as e:
            b.load_case_cell_components(0, NAMES)
        assert e.value.code == BAD_STATE
        k, status, size = b.load_case_info()
        assert k == 8 and size == 0 and status.shape == (8,)
        assert raw_images(b, size=0) == raw_images(b, size=8193) == BAD_ARG
        assert raw_images(b, aff=None) == raw_images(b, out=None) == BAD_ARG
        assert raw_images(b) == 0
        assert raw_components(b, n=0) == raw_components(b, n=5) == BAD_ARG
        assert raw_components(b, field_ids=np.array([0, 1, 4, 2], np.int32)) == BAD_ARG
        assert lib.fea_batch_load_case_strain_stress(b.h, -1, None, None) == BAD_ARG
        assert raw_components(b) == 0
        assert outputs_of_cases(b, affine)["strain", 0].shape[0] == 8

        assert b.load_case_info()[2] == SIZE
        res = b.solve_load_cases(loads[[2, 5, 3]], RTOL, MAX_ITER)   # a later call replaces what was kept
        k, status, size = b.load_case_info()
        assert k == 3 and status.tobytes() == res.status.tobytes() and size == SIZE
        three = outputs_of_cases(b, affine)
        assert three["images"].shape[0] == 3 and three["strain", 0].shape[0] == 3
        for i, k in enumerate([2, 5, 3]):
            assert_case_is_single(three, i, outputs_of_single(ctx, s, declare, loads[k], affine), ("replaced", i))
        assert res.status[1] == SAMPLE_BREAKDOWN

        after = b.download(images=True)                  # the batch's own results are untouched
        for f in ("u", "ranges", "iters", "relres", "status", "images"):
            assert np.asarray(getattr(after, f)).tobytes() == np.asarray(getattr(own, f)).tobytes(), f
        again = b.rasterize_cell_components(-1, NAMES, SCALE)
        for nm in NAMES:
            assert np.array_equal(again[0][nm], own_components[0][nm]) and same_floats(again[1][nm], own_components[1][nm])
