#!/usr/bin/env python
"""Multigrid from background grids (fea_batch_set_grid_hierarchy) against block-Jacobi CG and, where the mesh has
one, the caller-supplied hierarchy, all in one process, alternating, after one warm-up solve of each:

  * cantilever-L4, jittered (``workload.jittered_case``); caller hierarchy: the unjittered L0..L3 as coarse meshes;
  * one plate (``workload.plate_meshes``, seed 1) at h = 0.000625, 1.32 M vertices; caller hierarchy: the same
    geometry at h = 0.00125 .. 0.02 as coarse meshes;
  * gusset-L3 given as a plain mesh; caller hierarchy: its uniform refinement (set_refinement(3));
  * cantilever-L4; caller hierarchy: set_refinement(4).

    python tools/mg_grid_solve.py [--reps 3] [--out profiles/logs/r07_mg_grid_solve.jsonl]

The grid hierarchy gets round(log4(n_vertices / 2000)) levels (clamped to 1..8): its coarsest grid then has a
few thousand vertices, about what the caller hierarchies' coarsest meshes have.  One JSON line per (path, mesh):
solve ms from CUDA events around fea_batch_solve (median and every repetition), assemble ms (declaration +
fea_batch_assemble), outer iterations, V-cycle ms per level (level 0 = coarse solves), level sizes and the most
2x2 blocks in a row of each level, status, rel-L2 of u against block-Jacobi CG, and the device name and power
limit."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # the timing itself does not depend on it
        return "unknown (%s)" % e, "unknown"


def grid_levels(n_vertices):
    return int(min(8, max(1, round(math.log(max(n_vertices, 1) / 2000.0, 4)))))


def run(ctx, packed, declare, shapes):
    """(assemble ms, solve ms, result, stats, levels, row lengths) of one fresh batch; declare = None: block-Jacobi"""
    with ctx.create_batch(packed) as b:
        ctx.event_record(0)
        if declare is not None:
            declare(b)
        b.assemble()
        ctx.event_record(1)
        b.solve(1e-10, 400000)
        ctx.event_record(2)
        ctx.synchronize()
        t_asm, t_solve = ctx.event_elapsed_ms(0, 1), ctx.event_elapsed_ms(1, 2)
        r = b.download()
        lv = b.mg_levels() if declare is not None else None
        rows = None
        if shapes and lv is not None:
            rows = [int(np.diff(b.level_csr(l).indptr).max()) // 2 for l in range(len(lv))]
        return t_asm, t_solve, r, b.stats(), lv, rows


def cases():
    from fea_diffusion_b200 import pack
    from fea_diffusion_b200.host import ProblemSetup
    from fea_diffusion_b200.workload import jittered_case, large_case, plate_condition, plate_meshes
    s, _ = jittered_case("cantilever", 4)
    coarse = pack([large_case("cantilever", l)[0].sample for l in range(4)])
    yield "cantilever-L4-jittered", pack([s]), ("coarse_meshes", lambda b: b.set_coarse_meshes(coarse))
    t = time.time()
    sizes = [0.02, 0.01, 0.005, 0.0025, 0.00125, 0.000625]
    meshes, ptags, ltags = plate_meshes(1, sizes)
    kw = plate_condition(ptags, ltags)
    smp = [ProblemSetup(c, n, **kw).sample for c, n in meshes]
    print(json.dumps({"plate_mesh_vertices": [len(x.coors) for x in smp], "h": sizes,
                      "host_mesh_s": round(time.time() - t, 1)}), flush=True)
    pc = pack(smp[:-1])
    yield "plate-h0.000625", pack(smp[-1:]), ("coarse_meshes", lambda b: b.set_coarse_meshes(pc))
    yield "gusset-L3", pack([large_case("gusset", 3)[0].sample]), ("refinement", lambda b: b.set_refinement(3))
    yield "cantilever-L4", pack([large_case("cantilever", 4)[0].sample]), ("refinement", lambda b: b.set_refinement(4))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from fea_diffusion_b200 import Context
    name_dev, power = device_info()
    ctx = Context(0)
    lines = []
    for mesh, packed, (caller_kind, caller) in cases():
        levels = grid_levels(packed.n_vertices)
        paths = {"grid_hierarchy": lambda b: b.set_grid_hierarchy(levels), "block_jacobi": None,
                 "caller_" + caller_kind: caller}
        acc = {p: [] for p in paths}
        for rep in range(a.reps + 1):          # rep 0 warms every path up
            for p, declare in paths.items():
                acc[p].append(run(ctx, packed, declare, rep == a.reps) + (rep,))
        u_ref = acc["block_jacobi"][-1][2].u
        med = {}
        for p in paths:
            timed = [x for x in acc[p] if x[-1] > 0]
            t_asm, t_solve, r, st, lv, rows, _ = timed[-1]
            solves = [round(x[1], 3) for x in timed]
            med[p] = float(np.median(solves))
            line = {"path": p, "mesh": mesh, "n_vertices": int(packed.n_vertices),
                    "solve_ms_median": med[p], "solve_ms": solves,
                    "assemble_ms": [round(x[0], 3) for x in timed],
                    "outer_iterations": int(st["iterations"]), "status": int(r.status[0]), "relres": float(r.relres[0]),
                    "rel_l2_vs_block_jacobi": float(np.linalg.norm(r.u - u_ref) / np.linalg.norm(u_ref)),
                    "device": name_dev, "power_limit": power}
            if lv is not None:
                line["level_ms"] = [round(x["vcycle_ms"], 3) for x in lv]
                line["level_vertices"] = [int(x["n_vertices"]) for x in lv]
                line["level_dofs"] = [int(x["n_active_dofs"]) for x in lv]
                line["level_max_row_blocks"] = rows
                line["lambda_max"] = [round(x["lambda_max"], 4) for x in lv]
            print(json.dumps(line), flush=True)
            lines.append(line)
        line = {"mesh": mesh, "grid_levels": levels,
                "speedup_grid_over_block_jacobi": round(med["block_jacobi"] / med["grid_hierarchy"], 2),
                "grid_over_caller_time": round(med["grid_hierarchy"] / med["caller_" + caller_kind], 2),
                "device": name_dev, "power_limit": power}
        print(json.dumps(line), flush=True)
        lines.append(line)
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
