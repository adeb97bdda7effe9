"""CPU-side checks: the C-ABI library builds, loads and exports exactly what include/fea_b200.h
declares (no compute calls without a GPU); the host set-up logic agrees with the oracle."""
import os
import re
import subprocess

import numpy as np
import pytest

import cases
from fea_diffusion_b200 import _capi, host, imaging
from fea_diffusion_b200.solver import pack
from oracle import mesh_io
from oracle import raster_oracle as ro
from oracle.fea_oracle import OracleProblem

ROOT = cases.ROOT


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    return _capi.load_library()


def test_header_symbols_all_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "fea_b200.h")).read()
    declared = sorted(set(re.findall(r"^(?:int|const char\*)\s+(fea_[a-z_0-9]+)\s*\(", hdr, flags=re.M)))
    assert declared == sorted(_capi.EXPORTS)
    out = subprocess.run(["nm", "-D", "--defined-only", _capi.LIB_PATH], capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    for name in declared:
        assert name in exported, name
        assert getattr(lib, name) is not None


def test_version_call(lib):
    import ctypes as C
    a, b = C.c_int(-1), C.c_int(-1)
    assert lib.fea_version(C.byref(a), C.byref(b)) == 0
    assert (a.value, b.value) == (0, 3)


def test_library_is_sm100a_only():
    out = subprocess.run(["cuobjdump", "--list-elf", _capi.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_missing_library_fails_loudly(tmp_path):
    with pytest.raises(_capi.FeaError):
        _capi.load_library(str(tmp_path / "nope.so"))


@pytest.mark.parametrize("make", [cases.composite, lambda: cases.composite(False), cases.quad_plate])
def test_host_setup_matches_oracle(make):
    setup, orc = make()
    s = setup.sample
    assert np.array_equal(s.fixed.astype(bool), orc.fixed_vertex)
    assert np.array_equal(s.rhs, orc.load)
    assert np.array_equal(s.cell_region.astype(int), orc.cell_region.astype(int))
    assert np.array_equal(s.D, orc.D)
    assert setup.magnitudes_lines == orc.magnitudes_lines
    assert setup.materials_lines == orc.materials_lines
    for k, v in orc.region_vertices.items():
        assert np.array_equal(np.sort(setup.regions[k]), np.sort(v)), k
    fl, empty = host.floating_components(s)
    c = orc.classify()
    assert (fl, empty) == (c["floating_components"], c["empty_rows"])


def test_edge_force_text_and_magnitude():
    setup, orc = cases.composite()
    line = [l for l in setup.magnitudes_lines if l.startswith("EdgeForce0")][0]
    nv = len(setup.regions["EdgeForce0"])
    assert nv > 1
    assert line == "EdgeForce0:%s" % str((-300 / nv, 120 / nv))
    assert setup.n_terms == 2  # F2: load applied once per material term


def test_overlapping_material_regions_sum_their_D():
    """A-18: round coordinates can put a cell in two regions; K_e is linear in D so the cell gets
    the summed matrix -- equals the oracle's sum of per-region assemblies."""
    co = np.array([[0, 0], [1, 0], [1, 1], [0, 1], [2, 0], [2, 1.0]])
    cn = np.array([[0, 1, 2], [0, 2, 3], [1, 4, 5], [1, 5, 2]], np.int32)
    mats = {(100.0, 0.3): [(0, 0), (1, 0), (1, 1), (0, 1)], (50.0, 0.2): [(1, 0), (2, 0), (2, 1), (1, 1), (0, 0)]}
    kw = dict(force_vertex_tags_magnitudes=[(6, (1, 2))], constraints_vertex_tags=[1, 4],
              material_properties_to_vertices=mats)
    setup = host.ProblemSetup(co, cn, **kw)
    orc = OracleProblem(co, cn, **kw)
    assert orc.overlap_cells() > 0
    from oracle.fea_oracle import assemble_csr, element_stiffness
    s = setup.sample
    Ke = element_stiffness(orc.coors, orc.conn, s.D[np.maximum(s.cell_region, 0)])
    A = assemble_csr(len(co), orc.conn, Ke, s.cell_region, s.fixed.astype(bool))
    B = orc.stiffness()
    assert np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices)
    assert np.allclose(A.data, B.data, rtol=1e-14, atol=1e-12)


def test_read_mesh_matches_oracle_reader(tmp_path):
    p = tmp_path / "t.mesh"
    p.write_text(" MeshVersionFormatted 2\n Dimension\n 3\n Vertices\n 4\n 0 0 0 1\n 1 0 0 2\n"
                 " 1 0.5 0 3\n 0 0.5 0 4\n Edges\n 1\n 1 2 1\n Triangles\n 2\n 1 2 3 1\n 1 3 4 1\n End\n")
    co, cn = host.read_mesh(str(p))
    m = mesh_io.read_medit(str(p))
    assert np.array_equal(co, m["coors"]) and np.array_equal(cn, m["conn"])
    assert cn.dtype == np.int32 and co.shape == (4, 2)


def test_vtk_roundtrip(tmp_path, golden):
    co, cn = golden["cantilever_coors"], golden["cantilever_vtk_cells"]
    p = tmp_path / "o.vtk"
    mesh_io.write_vtk_legacy(str(p), co, cn,
                             point_data={"u": golden["cantilever_u"], "node_groups": golden["cantilever_node_groups"]},
                             cell_data={"mat_id": golden["cantilever_mat_id"]})
    v = mesh_io.read_vtk_legacy(str(p))
    assert np.array_equal(v["points"][:, :2], co) and np.array_equal(v["cells"], cn)
    assert np.array_equal(v["point_data"]["u"], golden["cantilever_u"])


@pytest.mark.parametrize("bbox", [(0, 0.4, 1, 0.6), (0, 0, 1, 1), (0, 0, 0.37, 1.0), (0.0, 0.0875, 1.0, 0.9125)])
@pytest.mark.parametrize("size", [64, 512])
def test_imaging_closed_form_matches_oracle(bbox, size):
    W, b = imaging.plate_window(bbox, size)
    assert (W, b) == ro.closed_form_window(bbox, size)
    assert np.array_equal(imaging.crop_affine(bbox, W, b), np.array(ro.pixel_affine(bbox, W, b)))
    assert abs((b[2] - b[0]) - size) <= 2


def test_pack_layout():
    s1, _ = cases.cantilever()
    s2, _ = cases.quad_plate()
    with pytest.raises(ValueError):
        pack([s1.sample, s2.sample])  # mixed cell types
    p = pack([s1.sample, s1.sample])
    assert p.vtx_off.tolist() == [0, 2464, 4928] and p.cell_off[-1] == 2 * 4686
    assert p.conn.dtype == np.int32 and p.fixed.dtype == np.uint8 and p.cell_region.dtype == np.int8
    assert p.desc.n_samples == 2 and p.desc.nodes_per_cell == 3


def test_every_context_option_is_documented_in_the_header():
    """fea_ctx_set_int accepts exactly the five options that select a path real inputs also reach
    (csrc/fea_api.cu), and include/fea_b200.h describes each of them."""
    import re
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    src = open(os.path.join(root, "fea_diffusion_b200", "csrc", "fea_api.cu")).read()
    body = src[src.index("int fea_ctx_set_int("):]
    body = body[:body.index("\n}\n")]
    keys = set(re.findall(r'strcmp\(key, "([a-z_]+)"\)', body))
    assert keys == {"pcg_path", "cluster_min", "cluster_halo_cap", "row_order", "refine_rounds"}
    header = open(os.path.join(root, "include", "fea_b200.h")).read()
    missing = [k for k in sorted(keys) if '"%s"' % k not in header]
    assert not missing, missing


def test_arena_device_addresses_and_descriptor_rebasing():
    """Host logic of the pipelined upload (no GPU): arrays carved from a PinnedArena map to the same offsets of
    its device copy, arrays from elsewhere do not; PackedConditions.use_device_copy rebases exactly the three
    big arrays of the descriptor (xy, conn, mat_coords) and nothing else."""
    from fea_diffusion_b200.solver import PackedConditions, PinnedArena

    class FakeCtx:                      # the two calls PinnedArena makes on a context
        def pinned_empty(self, shape, dtype):
            return np.empty(shape, dtype)

        def device_alloc(self, n):
            self.n = n
            return 0x7000_0000_0000

        def device_upload(self, dev, host, nbytes):
            self.uploaded = (dev, nbytes)

    ctx = FakeCtx()
    arena = PinnedArena(ctx, 1 << 20)
    co, cn = cases.small_plate() if hasattr(cases, "small_plate") else (np.array([[0., 0.], [1., 0.], [0., 1.], [1., 1.]]),
                                                                         np.array([[0, 1, 2], [1, 3, 2]], np.int32))
    kw = dict(force_vertex_tags_magnitudes=[(2, (1.0, 0.0))], constraints_vertex_tags=[1, 3],
              material_properties_to_vertices={(210000.0, 0.3): np.asarray(co, float)})
    pc = PackedConditions([(co, cn)], [(0, kw), (0, kw)], alloc=arena.empty)
    host_ptrs = {f: getattr(pc.desc, f) for f, _ in pc.desc._fields_}
    assert arena.device_address(pc.xy) is None                      # nothing uploaded yet
    arena.upload(ctx)
    assert ctx.uploaded == (0x7000_0000_0000, arena.off) and arena.spilled == 0
    base = arena.buf.ctypes.data
    for a in (pc.xy, pc.conn, pc.mat_coords):
        assert arena.device_address(a) == 0x7000_0000_0000 + (a.ctypes.data - base)
    assert arena.device_address(np.zeros(4)) is None and arena.device_address(pc.mesh_vtx_off) is None
    pc.use_device_copy(arena)
    for f, _ in pc.desc._fields_:
        v = getattr(pc.desc, f)
        if f in ("xy", "conn", "mat_coords"):
            assert v == 0x7000_0000_0000 + (getattr(pc, f).ctypes.data - base), f
        else:
            assert v == host_ptrs[f], f
