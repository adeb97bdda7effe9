#!/usr/bin/env python
"""The direct coarsest-level solver (fea_batch_set_coarse_solver(b, FEA_COARSE_DIRECT)) against the default
block-Jacobi CG coarse solve, on every hierarchy kind, in one process, the two paths alternating, after one warm-up
of each:

  * cantilever-L4, refinement (set_refinement(4));
  * cantilever-L4 jittered and the plate at h = 0.000625 (seed 1), coarse meshes (the unjittered L0..L3; the plate
    at h = 0.00125 .. 0.02);
  * cantilever-L4, gusset-L3 and the same plate, grid hierarchy with round(log4(n_vertices / 2000)) levels.

    python tools/mg_direct_coarse.py [--reps 3] [--out profiles/logs/r08_mg_direct_coarse.jsonl]

One JSON line per (path, row): assemble ms (declaration + fea_batch_assemble, CUDA events), factor ms (the dense
build, Cholesky and inversion, from fea_batch_get_coarse_info), solve ms of fea_batch_solve (median and every
repetition), outer iterations, V-cycle ms per level (level 0 = coarse solves), level-0 DOFs, smallest pivot, the
solve ms of 8 load cases in one fea_batch_solve_load_cases call, rel-L2 of u between the two paths, and the device
name and power limit as read."""
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

RTOL, MAX_ITER = 1e-10, 400


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


def eight_loads(s):
    """The model's load scaled, mirrored and restricted to halves of the free vertices: 8 distinct loads."""
    free = np.flatnonzero(~s.fixed.astype(bool))
    out = []
    for k in range(8):
        f = s.rhs * (1.0 + 0.25 * k)
        if k % 2:
            f = f[:, ::-1].copy()
        if k >= 4:
            g = np.zeros_like(f)
            half = free[(free % 2) == (k % 2)]
            g[half] = f[half]
            f = g
        out.append(f)
    return np.ascontiguousarray(np.stack(out))


def run(ctx, packed, declare, solver, loads):
    with ctx.create_batch(packed) as b:
        ctx.event_record(0)
        declare(b)
        b.set_coarse_solver(solver)
        b.assemble()
        ctx.event_record(1)
        b.solve(RTOL, MAX_ITER)
        ctx.event_record(2)
        ctx.synchronize()
        t_asm, t_solve = ctx.event_elapsed_ms(0, 1), ctx.event_elapsed_ms(1, 2)
        r = b.download()
        lv, info, st = b.mg_levels(), b.coarse_info(), b.stats()
        lc = b.solve_load_cases(loads, RTOL, MAX_ITER)
        return dict(asm=t_asm, solve=t_solve, u=r.u, status=int(r.status[0]), iters=int(st["iterations"]), lv=lv,
                    info=info, cases_ms=float(lc.stats["solve_ms"]), cases_iters=lc.iters.tolist(),
                    cases_converged=int(lc.stats["n_converged"]))


def rows():
    from fea_diffusion_b200 import pack
    from fea_diffusion_b200.host import ProblemSetup
    from fea_diffusion_b200.workload import jittered_case, large_case, plate_condition, plate_meshes
    cant = large_case("cantilever", 4)[0].sample
    yield "cantilever-L4", "refinement", cant, lambda b: b.set_refinement(4)
    s, _ = jittered_case("cantilever", 4)
    coarse = pack([large_case("cantilever", l)[0].sample for l in range(4)])
    yield "cantilever-L4-jittered", "coarse_meshes", s, lambda b: b.set_coarse_meshes(coarse)
    t = time.time()
    sizes = [0.02, 0.01, 0.005, 0.0025, 0.00125, 0.000625]
    meshes, ptags, ltags = plate_meshes(1, sizes)
    kw = plate_condition(ptags, ltags)
    smp = [ProblemSetup(c, n, **kw).sample for c, n in meshes]
    print(json.dumps({"plate_mesh_vertices": [len(x.coors) for x in smp], "h": sizes,
                      "host_mesh_s": round(time.time() - t, 1)}), flush=True)
    pc = pack(smp[:-1])
    plate = smp[-1]
    yield "plate-h0.000625", "coarse_meshes", plate, lambda b: b.set_coarse_meshes(pc)
    for name, smpl in (("cantilever-L4", cant), ("gusset-L3", large_case("gusset", 3)[0].sample), ("plate-h0.000625", plate)):
        levels = grid_levels(len(smpl.coors))
        yield name, "grid", smpl, (lambda lv: lambda b: b.set_grid_hierarchy(lv))(levels)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from fea_diffusion_b200 import Context, pack
    name_dev, power = device_info()
    ctx = Context(0)
    lines = []
    for mesh, kind, s, declare in rows():
        packed, loads = pack([s]), eight_loads(s)
        acc = {"cg": [], "direct": []}
        for rep in range(a.reps + 1):          # rep 0 warms both paths up
            for p in acc:
                acc[p].append(run(ctx, packed, declare, p, loads))
        med = {}
        for p in acc:
            timed = acc[p][1:]
            last = timed[-1]
            med[p] = {k: float(np.median([x[k] for x in timed])) for k in ("asm", "solve", "cases_ms")}
            med[p]["factor"] = float(np.median([x["info"]["factor_ms"] for x in timed]))
            other = acc["direct" if p == "cg" else "cg"][-1]["u"]
            line = {"path": p, "hierarchy": kind, "mesh": mesh, "n_vertices": int(len(s.coors)),
                    "assemble_ms_median": round(med[p]["asm"], 3), "assemble_ms": [round(x["asm"], 3) for x in timed],
                    "factor_ms_median": round(med[p]["factor"], 3),
                    "solve_ms_median": round(med[p]["solve"], 3), "solve_ms": [round(x["solve"], 3) for x in timed],
                    "outer_iterations": last["iters"], "status": last["status"],
                    "level_ms": [round(x["vcycle_ms"], 3) for x in last["lv"]],
                    "level_dofs": [int(x["n_active_dofs"]) for x in last["lv"]],
                    "coarse_n": int(last["info"]["n"]), "min_pivot": last["info"]["min_pivot"],
                    "inverse_bytes": int(last["info"]["bytes"]),
                    "rel_l2_u_vs_other_path": float(np.linalg.norm(last["u"] - other) / np.linalg.norm(other)),
                    "cases8_solve_ms_median": round(med[p]["cases_ms"], 3), "cases8_outer_iterations": last["cases_iters"],
                    "cases8_converged": last["cases_converged"], "device": name_dev, "power_limit": power}
            print(json.dumps(line), flush=True)
            lines.append(line)
        line = {"hierarchy": kind, "mesh": mesh,
                "direct_over_cg_solve": round(med["direct"]["solve"] / med["cg"]["solve"], 3),
                "direct_over_cg_assemble_plus_solve": round((med["direct"]["asm"] + med["direct"]["solve"]) /
                                                            (med["cg"]["asm"] + med["cg"]["solve"]), 3),
                "direct_over_cg_cases8": round(med["direct"]["cases_ms"] / med["cg"]["cases_ms"], 3),
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
