#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ from a checkout of the reference project
(namanxkumar/fea-diffusion):
    python tests/golden/make_golden.py <reference checkout>

Only DATA artefacts are converted (meshes, sfepy's committed fp64 ``u`` outputs,
committed PNG renders, text-format samples, log pins) -- no reference source.
Sources (relative to the checkout, SURVEY.md App. B):
  applications/cantilever/cantilever.{mesh,vtk}, displacement_[xy].png, outline.png
  applications/shearblade/shearblade.{mesh,vtk}, displacement_[xy].png, outline.png
  applications/gusset/gusset.mesh
  applications/composite/test.mesh, {magnitudes,materials,ranges}.txt
"""
import hashlib
import json
import os
import sys

import numpy as np
from PIL import Image

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
from oracle.mesh_io import read_medit, read_vtk_legacy  # noqa: E402

REF = sys.argv[1] if len(sys.argv) > 1 else os.environ.get("FEA_REFERENCE_DIR", "")


def sha16(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest()[:16]


def main():
    out = {}
    meta = {}
    for name in ("cantilever", "shearblade"):
        d = os.path.join(REF, "applications", name)
        m = read_medit(os.path.join(d, name + ".mesh"))
        v = read_vtk_legacy(os.path.join(d, name + ".vtk"))
        out[name + "_coors"] = m["coors"]
        out[name + "_conn"] = m["conn"]
        out[name + "_vtk_points"] = v["points"]
        out[name + "_vtk_cells"] = v["cells"].astype(np.int32)
        out[name + "_u"] = v["point_data"]["u"]
        out[name + "_node_groups"] = v["point_data"]["node_groups"].astype(np.int64)
        out[name + "_mat_id"] = v["cell_data"]["mat_id"].astype(np.int64)
        meta[name] = dict(mesh_sha=sha16(os.path.join(d, name + ".mesh")),
                          vtk_sha=sha16(os.path.join(d, name + ".vtk")))
        for png in ("displacement_x", "displacement_y", "outline"):
            im = np.array(Image.open(os.path.join(d, png + ".png")).convert("RGB"))
            out["%s_png_%s" % (name, png)] = im
    m = read_medit(os.path.join(REF, "applications/gusset/gusset.mesh"))
    out["gusset_coors"], out["gusset_conn"] = m["coors"], m["conn"]
    meta["gusset"] = dict(mesh_sha=sha16(os.path.join(REF, "applications/gusset/gusset.mesh")))
    m = read_medit(os.path.join(REF, "applications/composite/test.mesh"))
    out["composite_coors"], out["composite_conn"] = m["coors"], m["conn"]
    meta["composite"] = dict(mesh_sha=sha16(os.path.join(REF, "applications/composite/test.mesh")))
    # committed dataset images of the composite condition (the real datagen pipeline at image_size 512):
    # pins for the window sizing, crop and the region / input renders (SURVEY A-16, section 8f rank 4)
    for png in ("input", "outline", "regions_MaterialRegion0", "regions_MaterialRegion1", "regions_VertexForce0",
                "regions_VertexConstraint0"):
        im = np.array(Image.open(os.path.join(REF, "applications/composite", png + ".png")).convert("L"))
        out["composite_png_" + png] = im
    for t in ("magnitudes", "materials", "ranges"):
        meta["composite_" + t] = open(os.path.join(REF, "applications/composite", t + ".txt")).read()
    # log pins (file:line in SURVEY.md section 8c)
    meta["pins"] = dict(
        shearblade=dict(shape=10466, nnz=144084, r0=3.001666e+03,
                        src="test_nbs/generateapplication.ipynb:130,133,140"),
        composite=dict(cells=19307, shape=19672, nnz=270712, r0=8.000000e+02,
                       src="applications/composite/datagenapplication.ipynb:331,384,387,420"),
        cantilever=dict(n=4844, nnz=65896, fixed=42, src="SURVEY.md App. B (oracle-derived size)"),
    )
    # sfepy's displacements in a file of their own, which keeps each file under 1 MB
    np.savez_compressed(os.path.join(HERE, "reference_u.npz"), **{k: out.pop(k) for k in ("cantilever_u", "shearblade_u")})
    np.savez_compressed(os.path.join(HERE, "fixtures.npz"), **out)
    with open(os.path.join(HERE, "fixtures.json"), "w") as f:
        json.dump(meta, f, indent=1)
    print("wrote", os.path.join(HERE, "fixtures.npz"),
          os.path.getsize(os.path.join(HERE, "fixtures.npz")) // 1024, "KiB")


if __name__ == "__main__":
    main()
