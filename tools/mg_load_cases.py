#!/usr/bin/env python
"""Several load cases in one multigrid call (fea_batch_solve_load_cases) against one fea_batch_solve per case,
on three large meshes, both ways in one process, alternating, after one warm-up of each:

  * cantilever-L4 (``workload.large_case``), hierarchy ``set_refinement(4)``;
  * cantilever-L4, jittered (``workload.jittered_case``), coarse levels the unjittered L0..L3;
  * one plate (``workload.plate_meshes``, seed 1) at h = 0.000625, coarse levels the same geometry at
    h = 0.00125 .. 0.02, clamped on one edge and loaded at a corner (``workload.plate_condition``).

    python tools/mg_load_cases.py [--reps 3] [--out profiles/logs/r05_mg_load_cases.jsonl]

The 8 loads of a mesh: its own load, a horizontal point load at the free vertex farthest right, a load on the
right edge, and five seeded random loads on every free vertex.  A call with K cases solves the first K.  The K
single solves run on K batches created with those loads (assembled once, outside the timing).

One JSON line per (mesh, K): ms per call and per case (CUDA events around the call, which include copying the
loads in and u out through pageable host memory; median of ``--reps``), the call's solve ms without those copies
(``stats["solve_ms"]``, the span fea_batch_solve's solve_ms covers), the
sum of the K single solves' ms (fea_batch_solve, events) and the median single solve, outer iterations per
case, V-cycle ms per level of the call and of one single solve (level 0 = coarse solves), whether every case
is bit-identical to its single solve, and the device name and power limit."""
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


def eight_loads(s):
    free = ~s.fixed.astype(bool)
    x = s.coors[:, 0]
    point = np.zeros_like(s.rhs)
    point[np.flatnonzero(free)[np.argmax(x[free])]] = (1000.0, 0.0)
    edge = np.zeros_like(s.rhs)
    edge[free & (x >= x.max() - 1e-9 * (x.max() - x.min()))] = (0.0, -250.0)
    out = [s.rhs, point, edge]
    for seed in range(5):
        r = np.zeros_like(s.rhs)
        r[free] = np.random.default_rng(seed).uniform(-100.0, 100.0, (int(free.sum()), 2))
        out.append(r)
    return np.ascontiguousarray(np.stack(out))


def cases():
    from fea_diffusion_b200 import pack
    from fea_diffusion_b200.host import ProblemSetup
    from fea_diffusion_b200.workload import jittered_case, large_case, plate_condition, plate_meshes
    s = large_case("cantilever", 4)[0].sample
    yield "cantilever-L4", s, lambda b: b.set_refinement(4)
    coarse = pack([large_case("cantilever", l)[0].sample for l in range(4)])
    s, _ = jittered_case("cantilever", 4)
    yield "cantilever-L4-jittered", s, lambda b: b.set_coarse_meshes(coarse)
    t = time.time()
    sizes = [0.02, 0.01, 0.005, 0.0025, 0.00125, 0.000625]
    meshes, ptags, ltags = plate_meshes(1, sizes)
    kw = plate_condition(ptags, ltags)
    smp = [ProblemSetup(c, n, **kw).sample for c, n in meshes]
    print(json.dumps({"plate_mesh_vertices": [len(x.coors) for x in smp], "h": sizes,
                      "host_mesh_s": round(time.time() - t, 1)}), flush=True)
    pc = pack(smp[:-1])
    yield "plate-h0.000625", smp[-1], lambda b: b.set_coarse_meshes(pc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from fea_diffusion_b200 import Context, pack
    from fea_diffusion_b200.solver import Sample
    name_dev, power = device_info()
    ctx = Context(0)
    lines = []
    for mesh, s, declare in cases():
        loads = eight_loads(s)
        singles = []
        for k in range(len(loads)):
            b = ctx.create_batch(pack([Sample(s.coors, s.conn, s.cell_region, s.D, s.fixed, loads[k])]))
            declare(b)
            singles.append(b.assemble())
        batch = singles[0]   # its own load is case 0: the load-case calls run on it as well

        def call(K):
            ctx.event_record(0)
            res = batch.solve_load_cases(loads[:K], 1e-10, 400000)
            ctx.event_record(1)
            return ctx.event_elapsed_ms(0, 1), res, batch.mg_levels(), res.stats["solve_ms"]

        def separate(K):
            out = []
            for b in singles[:K]:
                ctx.event_record(0)
                b.solve(1e-10, 400000)
                ctx.event_record(1)
                out.append((ctx.event_elapsed_ms(0, 1), b.download(), b.mg_levels()))
            return out

        for K in (1, 2, 4, 8):
            runs_call, runs_sep = [], []
            for rep in range(a.reps + 1):   # rep 0 warms both up (and builds the K-sample coarsest batch)
                runs_call.append(call(K))
                runs_sep.append(separate(K))
            runs_call, runs_sep = runs_call[1:], runs_sep[1:]
            t_call, res, lv_call, _ = runs_call[-1]
            sep = runs_sep[-1]
            bitwise = all(
                res.u[k].tobytes() == sep[k][1].u.tobytes() and res.ranges[k].tobytes() == sep[k][1].ranges[0].tobytes()
                and res.iters[k] == sep[k][1].iters[0] and res.relres[k].tobytes() == sep[k][1].relres[0].tobytes()
                and res.status[k] == sep[k][1].status[0] for k in range(K))
            call_ms = float(np.median([x[0] for x in runs_call]))
            solve_ms = float(np.median([x[3] for x in runs_call]))
            sep_ms = float(np.median([sum(y[0] for y in x) for x in runs_sep]))
            single_ms = float(np.median([y[0] for x in runs_sep for y in x]))
            line = {"mesh": mesh, "n_vertices": int(len(s.coors)), "K": K,
                    "call_ms_median": round(call_ms, 3), "call_ms": [round(x[0], 3) for x in runs_call],
                    "call_ms_per_case": round(call_ms / K, 3),
                    "separate_ms_median": round(sep_ms, 3), "single_solve_ms_median": round(single_ms, 3),
                    "call_over_single": round(call_ms / single_ms, 3),
                    "call_solve_ms_median": round(solve_ms, 3), "call_solve_over_single": round(solve_ms / single_ms, 3),
                    "outer_iterations": res.iters.tolist(), "status": res.status.tolist(),
                    "single_outer_iterations": [int(x[1].iters[0]) for x in sep],
                    "level_ms_call": [round(x["vcycle_ms"], 3) for x in lv_call],
                    "level_ms_single": [round(x["vcycle_ms"], 3) for x in sep[0][2]],
                    "bitwise_equal_to_single_solves": bool(bitwise),
                    "device": name_dev, "power_limit": power}
            print(json.dumps(line), flush=True)
            lines.append(line)
        for b in singles:
            b.destroy()
    ctx.close()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
