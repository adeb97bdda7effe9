#!/usr/bin/env python
"""Time the streaming PCG kernels on BASELINE config 3 (cantilever L4 by default), all systems kept active
(rtol = 0, ITERS iterations).
    python tools/tune_spmv_c3.py [mesh level [row_order,...]]"""
import os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fea_diffusion_b200 import Context, pack
from fea_diffusion_b200.workload import large_case
name, lv = (sys.argv[1], int(sys.argv[2])) if len(sys.argv) > 2 else ("cantilever", 4)
orders = [int(x) for x in sys.argv[3].split(",")] if len(sys.argv) > 3 else [3]
iters = int(os.environ.get("ITERS", "2048"))
setup, _ = large_case(name, lv)
packed = pack([setup.sample])
ctx = Context(0)
for order in orders:
    ctx.set_option("row_order", order)
    with ctx.create_batch(packed) as b:
        b.assemble()
        info = b.info()
        for _ in range(2):
            b.solve(0.0, iters)
        st = b.stats()
    nn, nnz = info["n_active_dofs"], info["nnz"]
    alg = 12 * nnz + 4 * (nn + 1) + 16 * nn
    print(json.dumps({"row_order": order, "spmv_ms": st["spmv_ms_avg"], "update_ms": st["update_ms_avg"],
                      "us_per_iter": 1e3 * st["solve_ms"] / iters, "alg_GBs": alg / st["spmv_ms_avg"] / 1e6}), flush=True)
ctx.close()
