#!/usr/bin/env python
"""Multigrid from coarser meshes of the same domain (fea_batch_set_coarse_meshes) against block-Jacobi CG on
two meshes that are no uniform refinement, both paths in one process, alternating, after one warm-up solve of
each:

  * cantilever-L4, jittered (``workload.jittered_case``), coarse levels the unjittered L0..L3;
  * one plate (``workload.plate_meshes``, seed 1) at h = 0.000625, coarse levels the same geometry at
    h = 0.00125 .. 0.02, clamped on one edge and loaded at a corner (``workload.plate_condition``).

    python tools/mg_nonnested_solve.py [--reps 3] [--out profiles/logs/mg_nonnested_solve.jsonl]

One JSON line per (path, mesh): solve ms from CUDA events around fea_batch_solve (median and all
repetitions), assemble ms (set_coarse_meshes + fea_batch_assemble for multigrid), outer iterations, V-cycle ms
per level (level 0 = coarse solves), status, rel-L2 between the two paths' u, and the device name and power
limit.  A last line per config-3 mesh (cantilever-L4, gusset-L3, uniform refinements) compares the
Galerkin operators of ``set_refinement`` with the rediscretised ones that ``set_coarse_meshes`` builds from the
same coarse meshes: outer iterations and solve ms of each (median of ``--reps`` after a warm-up)."""
import argparse
import json
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


def run(ctx, packed, coarse):
    """(assemble ms, solve ms, result, stats, levels) of one fresh batch; coarse = None: block-Jacobi CG."""
    with ctx.create_batch(packed) as b:
        ctx.event_record(0)
        if coarse is not None:
            b.set_coarse_meshes(coarse)
        b.assemble()
        ctx.event_record(1)
        b.solve(1e-10, 400000)
        ctx.event_record(2)
        ctx.synchronize()
        t_asm, t_solve = ctx.event_elapsed_ms(0, 1), ctx.event_elapsed_ms(1, 2)
        r = b.download()
        return t_asm, t_solve, r, b.stats(), (b.mg_levels() if coarse is not None else None)


def cases():
    from fea_diffusion_b200 import pack
    from fea_diffusion_b200.host import ProblemSetup
    from fea_diffusion_b200.workload import jittered_case, large_case, plate_condition, plate_meshes
    s, _ = jittered_case("cantilever", 4)
    yield "cantilever-L4-jittered", pack([s]), pack([large_case("cantilever", l)[0].sample for l in range(4)])
    t = time.time()
    sizes = [0.02, 0.01, 0.005, 0.0025, 0.00125, 0.000625]
    meshes, ptags, ltags = plate_meshes(1, sizes)
    kw = plate_condition(ptags, ltags)
    smp = [ProblemSetup(c, n, **kw).sample for c, n in meshes]
    print(json.dumps({"plate_mesh_vertices": [len(x.coors) for x in smp], "h": sizes,
                      "host_mesh_s": round(time.time() - t, 1)}), flush=True)
    yield "plate-h0.000625", pack(smp[-1:]), pack(smp[:-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from fea_diffusion_b200 import Context
    name_dev, power = device_info()
    ctx = Context(0)
    lines = []
    for mesh, packed, coarse in cases():
        acc = {True: [], False: []}
        for rep in range(a.reps + 1):          # rep 0 warms both paths up
            for mg in (True, False):
                acc[mg].append(run(ctx, packed, coarse if mg else None) + (rep,))
        u = {mg: acc[mg][-1][2].u for mg in (True, False)}
        diff = float(np.linalg.norm(u[True] - u[False]) / np.linalg.norm(u[False]))
        for mg in (True, False):
            timed = [x for x in acc[mg] if x[-1] > 0]
            t_asm, t_solve, r, st, lv, _ = timed[-1]
            solves = [round(x[1], 3) for x in timed]
            line = {"path": "multigrid_nonnested" if mg else "block_jacobi", "mesh": mesh,
                    "n_vertices": int(packed.n_vertices),
                    "solve_ms_median": float(np.median(solves)), "solve_ms": solves,
                    "assemble_ms": [round(x[0], 3) for x in timed],
                    "outer_iterations": int(st["iterations"]), "status": int(r.status[0]), "relres": float(r.relres[0]),
                    "rel_l2_between_paths": diff, "device": name_dev, "power_limit": power}
            if mg:
                line["level_ms"] = [round(x["vcycle_ms"], 3) for x in lv]
                line["level_vertices"] = [int(x["n_vertices"]) for x in lv]
                line["level_dofs"] = [int(x["n_active_dofs"]) for x in lv]
                line["lambda_max"] = [round(x["lambda_max"], 4) for x in lv]
            print(json.dumps(line), flush=True)
            lines.append(line)
        speed = np.median([x[1] for x in acc[False] if x[-1] > 0]) / np.median([x[1] for x in acc[True] if x[-1] > 0])
        print(json.dumps({"mesh": mesh, "speedup_mg_over_block_jacobi": round(float(speed), 2)}), flush=True)
    from fea_diffusion_b200 import pack
    from fea_diffusion_b200.workload import large_case
    for name, level in (("cantilever", 4), ("gusset", 3)):
        packed = pack([large_case(name, level)[0].sample])
        coarse = pack([large_case(name, l)[0].sample for l in range(level)])
        res, u = {}, {}
        for how in ("galerkin", "rediscretised"):
            runs = []
            for rep in range(a.reps + 1):
                with ctx.create_batch(packed) as b:
                    if how == "galerkin":
                        b.set_refinement(level)
                    else:
                        b.set_coarse_meshes(coarse)
                    r = b.assemble().solve(1e-10, 200).download()
                    runs.append((b.stats()["iterations"], b.stats()["solve_ms"], int(r.status[0]), r.u))
            res[how] = {"outer_iterations": runs[-1][0], "solve_ms_median": float(np.median([x[1] for x in runs[1:]])),
                        "status": runs[-1][2]}
            u[how] = runs[-1][3]
        res["rel_l2_between"] = float(np.linalg.norm(u["rediscretised"] - u["galerkin"]) / np.linalg.norm(u["galerkin"]))
        line = {"mesh": "%s-L%d" % (name, level), "coarse_operators": res, "device": name_dev, "power_limit": power}
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
