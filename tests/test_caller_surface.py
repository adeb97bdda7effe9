"""The reference's own caller against the drop-in surface (north_star: "datagen/generate.py and
generate_data.py drive it unchanged").  Every call, keyword and attribute that
the reference's datagen/generate.py:56-164 uses on FEAnalysis / MeshGenerator / the two utils
functions -- extracted from its source by tests/golden/make_caller_surface.py and committed as
tests/golden/caller_surface.json -- must bind against this package's classes; with a checkout of the
reference named by FEA_REFERENCE_DIR the fixture is re-derived and the reference's file itself is loaded
over the drop-in."""
import importlib.util
import inspect
import json
import os

import pytest

from fea_diffusion_b200.datagen import FEAnalysis, fea_analysis, mesh_generator, utils
from fea_diffusion_b200.datagen.generate import generate_data, load_reference_generate
from fea_diffusion_b200.datagen.mesh_generator import MeshGenerator

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("FEA_REFERENCE_DIR", "")


def committed():
    with open(os.path.join(HERE, "golden", "caller_surface.json")) as f:
        return json.load(f)


def binds(fn, sig, bound_method):
    """the call shape (n positional, these keywords) is accepted by fn"""
    params = inspect.signature(fn)
    args = [object()] * (sig["n_pos"] + (1 if bound_method else 0))
    params.bind(*args, **{k: object() for k in sig["keywords"]})


def test_every_use_the_reference_caller_makes_binds_to_the_dropin():
    s = committed()
    assert s["imports"] == {"fea_analysis": ["FEAnalysis"], "mesh_generator": ["MeshGenerator"],
                            "utils": ["find_image_bounds", "verify_directory"]}
    assert hasattr(fea_analysis, "FEAnalysis") and hasattr(mesh_generator, "MeshGenerator")
    for cls, name in ((FEAnalysis, "FEAnalysis"), (MeshGenerator, "MeshGenerator")):
        binds(cls.__init__, s[name]["init"], True)
        for m, sig in s[name]["methods"].items():
            assert callable(getattr(cls, m, None)), (name, m)
            binds(inspect.getattr_static(cls, m).__func__ if isinstance(inspect.getattr_static(cls, m), staticmethod)
                  else getattr(cls, m), sig, not isinstance(inspect.getattr_static(cls, m), staticmethod))
    for fn, sig in s["functions"].items():
        binds(getattr(utils, fn), sig, False)
    # attributes the caller reads are set by the constructor (fea_analysis.py:54 -> generate.py:135)
    src = inspect.getsource(FEAnalysis.__init__)
    for a in s["FEAnalysis"]["attributes"]:
        assert "self.%s" % a in src, a
    # same keyword surface and defaults as the reference's generate_data (generate.py:12-31)
    p = inspect.signature(generate_data).parameters
    assert [k for k in p][:17] == ["data_dir", "image_size", "num_plates", "start_plate", "conditions_per_plate", "mesh_size",
                                  "num_polygons_range", "points_per_polygon_range", "holes_per_polygon_range",
                                  "points_per_hole_range", "num_regions", "save_displacement", "save_strain", "save_stress",
                                  "num_steps_per_condition", "save_meshes", "wandb_inject_function"]
    assert p["num_steps_per_condition"].default == 11 and p["image_size"].default == 512 and p["mesh_size"].default == 1e-2


def test_constructor_signature_is_the_reference_one():
    """fea_analysis.py:32-48: positional order and defaults."""
    p = list(inspect.signature(FEAnalysis.__init__).parameters.values())
    names = [q.name for q in p if q.kind == q.POSITIONAL_OR_KEYWORD]
    assert names == ["self", "filename", "data_dir", "condition_dir", "force_vertex_tags_magnitudes",
                     "force_edges_tags_magnitudes", "constraints_vertex_tags", "constraints_edges_tags", "num_steps",
                     "save_meshes", "material_properties_to_vertices", "youngs_modulus", "poisson_ratio"]
    d = {q.name: q.default for q in p}
    assert (d["num_steps"], d["save_meshes"], d["material_properties_to_vertices"], d["youngs_modulus"], d["poisson_ratio"]) == \
        (11, False, None, 210000, 0.3)


@pytest.mark.skipif(not (REF and os.path.isfile(os.path.join(REF, "datagen", "generate.py"))), reason="needs a reference checkout (FEA_REFERENCE_DIR)")
def test_fixture_is_current_and_the_reference_file_loads_over_the_dropin():
    spec = importlib.util.spec_from_file_location("make_caller_surface", os.path.join(HERE, "golden", "make_caller_surface.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    with open(os.path.join(REF, "datagen", "generate.py")) as f:
        assert mod.surface(f.read()) == committed()
    fn = load_reference_generate(REF)              # the reference's own source, imports bound to this package
    m = inspect.getmodule(fn)
    assert m.FEAnalysis is FEAnalysis and m.MeshGenerator is MeshGenerator
    assert m.find_image_bounds is utils.find_image_bounds and m.verify_directory is utils.verify_directory
    assert os.path.samefile(inspect.getsourcefile(fn), os.path.join(REF, "datagen", "generate.py"))
