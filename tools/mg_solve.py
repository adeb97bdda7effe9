#!/usr/bin/env python
"""Multigrid-preconditioned against block-Jacobi CG on BASELINE config 3 (cantilever-L4, gusset-L3,
``workload.large_case``), both paths in one process, alternating, after one warm-up solve of each.

    python tools/mg_solve.py [--reps 3] [--out profiles/logs/mg_solve.jsonl]

One JSON line per (path, mesh): solve ms from CUDA events around fea_batch_solve (median and all
repetitions), outer iterations, multigrid ms per level (level 0 = coarse solves), set-up (assemble)
ms, rel-L2 against tests/golden/c3_lu.npz, and the device name and power limit."""
import argparse
import json
import os
import subprocess
import sys

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


def run(ctx, packed, levels, mg):
    """(assemble ms, solve ms, result, stats, levels) of one fresh batch."""
    with ctx.create_batch(packed) as b:
        if mg:
            b.set_refinement(levels)
        ctx.event_record(0)
        b.assemble()
        ctx.event_record(1)
        b.solve(1e-10, 400000)
        ctx.event_record(2)
        ctx.synchronize()
        t_asm, t_solve = ctx.event_elapsed_ms(0, 1), ctx.event_elapsed_ms(1, 2)
        r = b.download()
        return t_asm, t_solve, r, b.stats(), (b.mg_levels() if mg else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from fea_diffusion_b200 import Context, pack
    from fea_diffusion_b200.workload import large_case
    ref = np.load(os.path.join(ROOT, "tests", "golden", "c3_lu.npz"))
    name_dev, power = device_info()
    ctx = Context(0)
    lines = []
    for name, level in (("cantilever", 4), ("gusset", 3)):
        setup, n0 = large_case(name, level)
        packed = pack([setup.sample])
        g = ref["%s_L%d_u_coarse" % (name, level)]
        acc = {True: [], False: []}
        for rep in range(a.reps + 1):          # rep 0 warms both paths up
            for mg in (True, False):
                acc[mg].append(run(ctx, packed, level, mg) + (rep,))
        for mg in (True, False):
            timed = [x for x in acc[mg] if x[-1] > 0]
            t_asm, t_solve, r, st, lv, _ = timed[-1]
            solves = [round(x[1], 3) for x in timed]
            line = {"path": "multigrid" if mg else "block_jacobi", "mesh": "%s-L%d" % (name, level),
                    "n_dofs": int(ref["%s_L%d_n_dofs" % (name, level)]),
                    "solve_ms_median": float(np.median(solves)), "solve_ms": solves,
                    "assemble_ms": [round(x[0], 3) for x in timed],
                    "outer_iterations": int(st["iterations"]), "status": int(r.status[0]),
                    "rel_l2_vs_c3_lu": float(np.linalg.norm(r.u[:n0] - g) / np.linalg.norm(g)),
                    "device": name_dev, "power_limit": power}
            if mg:
                line["level_ms"] = [round(x["vcycle_ms"], 3) for x in lv]
                line["coarse_solve_ms"] = round(lv[0]["vcycle_ms"], 3)
                line["level_dofs"] = [int(x["n_active_dofs"]) for x in lv]
                line["lambda_max"] = [round(x["lambda_max"], 4) for x in lv]
            print(json.dumps(line), flush=True)
            lines.append(line)
        speed = np.median([x[1] for x in acc[False] if x[-1] > 0]) / np.median([x[1] for x in acc[True] if x[-1] > 0])
        print(json.dumps({"mesh": "%s-L%d" % (name, level), "speedup_mg_over_block_jacobi": round(float(speed), 2)}), flush=True)
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
