#!/usr/bin/env python
"""Cluster classes of a bench workload (by seed): systems, iterations and CTA-iterations per class, the longest
single solves, and the solve time -- to see what a batch's critical path is.
    python tools/class_probe.py [seed0] [plates]"""
import os, sys, json
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fea_diffusion_b200 import Context, pack
from fea_diffusion_b200.workload import build_workload
seed0 = int(sys.argv[1]) if len(sys.argv) > 1 else 0
plates = int(sys.argv[2]) if len(sys.argv) > 2 else 100
items, _ = build_workload(plates, 4, 64, seed0=seed0, workers=os.cpu_count() or 1)
ctx = Context(0)
packed = pack([it.setup.sample for it in items], alloc=ctx.pinned_empty)
with ctx.create_batch(packed) as b:
    b.assemble()
    ms = []
    for _ in range(4):
        b.solve(1e-10, 20000)
        ms.append(round(b.stats()["cluster_ms"], 2))
    r = b.download()
    rounds = b.refine_rounds()
nv = np.diff(packed.vtx_off)
rows = (nv + 127) // 128 * 128
cl = np.maximum(1, (rows + 2047) // 2048)
us_it = 3.9e-3   # ms per iteration, roughly
print(json.dumps({"seed0": seed0, "cluster_ms": ms, "iters_sum": int(r.iters.sum()), "iters_max": int(r.iters.max()),
                  "refined": int((rounds > 0).sum())}))
tot = float((r.iters * cl).sum())
for c in sorted(set(cl.tolist())):
    m = cl == c
    print("class %d: %3d systems  iterations mean %5.0f max %5d  CTA-iterations %.0f (%.1f %%)" %
          (c, m.sum(), r.iters[m].mean(), r.iters[m].max(), float((r.iters[m] * c).sum()), 100 * float((r.iters[m] * c).sum()) / tot))
print("ideal ms at 148 SMs x 3.8 us per CTA-iteration: %.1f" % (tot * 3.8e-3 / 148))
top = np.argsort(-r.iters)[:8]
print("longest solves:", [(int(i), int(r.iters[i]), int(nv[i]), int(cl[i]), int(rounds[i])) for i in top], "(sample, iterations, vertices, class, refinement rounds)")
