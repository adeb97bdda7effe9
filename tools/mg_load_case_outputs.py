#!/usr/bin/env python
"""Outputs of K = 8 load cases from one multigrid call (fea_batch_load_case_images / _strain_stress /
_cell_components) against 8 single batches created, assembled, solved and post-processed with the same loads,
both ways in one process, alternating, after one warm-up of each:

  * cantilever-L4 (``workload.large_case``), hierarchy ``set_refinement(4)``;
  * one plate (``workload.plate_meshes``, seed 1) at h = 0.000625 (1.32 M vertices), coarse levels the same
    geometry at h = 0.00125 .. 0.02 (``set_coarse_meshes``).

    python tools/mg_load_case_outputs.py [--reps 3] [--size 512] [--out profiles/logs/r06_mg_load_case_outputs.jsonl]

The meshes and the 8 loads are those of tools/mg_load_cases.py.  Post-processing is what a dataset sample gets:
the displacement images, the cell strain / stress (each cell's own D) and the four stress / strain component
images with their ranges (stress_region 0), at --size pixels with the camera of ``imaging.plate_window``.

One JSON line per mesh, medians of ``--reps`` (host clock; every call ends in a stream synchronise and includes
its copies to pageable host memory):
  * ``outputs_ms``: the three load-case output calls for the 8 cases;
  * ``single_outputs_ms``: the same outputs of the 8 single batches (fea_batch_rasterize +
    fea_batch_download_images, cell_strain_stress, rasterize_cell_components), summed; both columns copy the same
    bytes to the host (u came back with the solve on either side, outside these windows);
  * ``call_and_outputs_ms``: fea_batch_solve_load_cases of the 8 loads plus ``outputs_ms``;
  * ``singles_ms``: the 8 single batches end to end (create, declare, assemble, solve, download of u, ranges,
    iterations, relres and status as solve_load_cases returns them, post-process, destroy);
whether every output of every case is bit-identical to its single batch's, and the device name and power limit."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from mg_load_cases import cases, device_info, eight_loads  # noqa: E402

NAMES = ["stress_x", "stress_y", "strain_x", "strain_y"]


def camera(s, size):
    from fea_diffusion_b200.imaging import crop_affine, plate_window
    x, y = s.coors[:, 0], s.coors[:, 1]
    bbox = (x.min(), y.min(), x.max(), y.max())
    window, bounds = plate_window(bbox, size)
    return crop_affine(bbox, window, bounds)


def post_process(b, size, affine):
    """Outputs of a solved single batch, timed without its creation and solve: (ms, outputs).  It copies to the
    host exactly what the load-case output calls copy: no u, ranges or solve statistics (fea_batch_download), which
    the load-case path returns from the solve call."""
    from fea_diffusion_b200._capi import ptr
    images = np.empty((1, 2, size, size), np.uint8)
    t = time.perf_counter()
    b.rasterize(size, affine.reshape(1, 4), 1.0)
    b.ctx._check(b.ctx.lib.fea_batch_download_images(b.h, ptr(images)))
    strain, stress = b.cell_strain_stress(-1)
    comp_img, comp_rng = b.rasterize_cell_components(0, NAMES, 1.0)
    ms = 1e3 * (time.perf_counter() - t)
    return ms, (images[0], strain, stress, np.stack([comp_img[n][0] for n in NAMES]), np.stack([comp_rng[n][0] for n in NAMES]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from fea_diffusion_b200 import Context, pack
    from fea_diffusion_b200.solver import Sample
    name_dev, power = device_info()
    ctx = Context(0)
    lines = []
    for mesh, s, declare in cases():
        if mesh == "cantilever-L4-jittered":
            continue
        loads = eight_loads(s)
        affine = camera(s, a.size)
        batch = ctx.create_batch(pack([s]))
        declare(batch)
        batch.assemble()

        def load_cases():
            t = time.perf_counter()
            batch.solve_load_cases(loads, 1e-10, 400000)
            t1 = time.perf_counter()
            images = batch.load_case_images(a.size, affine, 1.0)
            strain, stress = batch.load_case_strain_stress(-1)
            comp_img, comp_rng = batch.load_case_cell_components(0, NAMES, 1.0)
            t2 = time.perf_counter()
            out = [(images[k], strain[k], stress[k], np.stack([comp_img[n][k] for n in NAMES]),
                    np.stack([comp_rng[n][k] for n in NAMES])) for k in range(len(loads))]
            return 1e3 * (t2 - t), 1e3 * (t2 - t1), out

        def singles():
            t = time.perf_counter()
            post_ms, out = 0.0, []
            for k in range(len(loads)):
                b = ctx.create_batch(pack([Sample(s.coors, s.conn, s.cell_region, s.D, s.fixed, loads[k])]))
                declare(b)
                b.assemble().solve(1e-10, 400000).download()   # u, as solve_load_cases returns it
                ms, o = post_process(b, a.size, affine)
                post_ms += ms
                out.append(o)
                b.destroy()
            return 1e3 * (time.perf_counter() - t), post_ms, out

        runs_lc, runs_single = [], []
        for rep in range(a.reps + 1):   # rep 0 warms both up (and builds the 8-sample coarsest batch)
            runs_lc.append(load_cases())
            runs_single.append(singles())
        runs_lc, runs_single = runs_lc[1:], runs_single[1:]
        got, want = runs_lc[-1][2], runs_single[-1][2]
        bitwise = all(x.tobytes() == y.tobytes() for k in range(len(loads)) for x, y in zip(got[k], want[k]))
        med = lambda xs: float(np.median(xs))  # noqa: E731
        line = {"mesh": mesh, "n_vertices": int(len(s.coors)), "n_cells": int(len(s.conn)), "K": len(loads),
                "image_size": a.size,
                "output_host_bytes": int(sum(x.nbytes for o in got for x in o)),   # either way, per window
                "outputs_ms": round(med([r[1] for r in runs_lc]), 3), "outputs_ms_runs": [round(r[1], 3) for r in runs_lc],
                "single_outputs_ms": round(med([r[1] for r in runs_single]), 3),
                "single_outputs_ms_runs": [round(r[1], 3) for r in runs_single],
                "call_and_outputs_ms": round(med([r[0] for r in runs_lc]), 3),
                "singles_ms": round(med([r[0] for r in runs_single]), 3),
                "bitwise_equal_to_single_batches": bool(bitwise),
                "device": name_dev, "power_limit": power}
        line["outputs_speedup"] = round(line["single_outputs_ms"] / line["outputs_ms"], 3)
        line["end_to_end_speedup"] = round(line["singles_ms"] / line["call_and_outputs_ms"], 3)
        print(json.dumps(line), flush=True)
        lines.append(line)
        batch.destroy()
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
