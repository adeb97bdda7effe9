#!/usr/bin/env python
"""bench.py -- plate-condition FEA solves/s on N B200s (BASELINE.json metric).

One "step" = one pass of the hot path over one batch of synthetic plate-condition samples:
assembly + Dirichlet elimination + block-Jacobi PCG solve (all load steps of a condition are t_k
multiples of one solve, SURVEY F5) + ranges + the two 64x64 displacement images.
Default workload = BASELINE.json configs[1]: 100 plates x 4 conditions x 10 loaded steps
(steps_per_condition 11), default mesh density, image_size 64.

  value : device-resident throughput (inputs already in HBM), CUDA events on the library stream
  e2e   : same metric through the one-call host-buffer C-ABI entry (fea_solve_batch): pinned host
          inputs -> H2D -> assemble/solve/raster -> D2H of u, ranges, images, every step
  roofline    : the dominant kernel (k_pcg_cluster launch group), algorithmic bytes / event-timed launch
  cpu_baseline: the CPU oracle (numpy + scipy SuperLU restatement of the reference path) timed on
                this box's host cores on a bounded sample; cpu_baseline_best = factor once + scale
  dataset_e2e : samples/s from in-memory meshes + condition dicts (tags, magnitudes, material
                coordinate lists): host packing, H2D, region selection / Dirichlet mask / load on the
                device (fea_batch_create_from_conditions), assemble, solve, raster of u and of every
                region, classifier, D2H -- everything but meshing and PNG/text encoding
  as_sampled  : the same path on the sampler's own condition distribution (a third singular, F4)
  c3 / c1     : BASELINE configs 3 (~1 M-DOF single solves) and 1 (one plate-condition through the
                drop-in FEAnalysis.calculate())

`--steps K` is the number of timed steps of value, e2e and dataset_e2e.  `--dump-outputs DIR` writes what the last
timed device-resident step computed (dump_outputs); the workload is seeded, so two builds run with the same
arguments can be compared output for output.

`--impl reference` times the reference's CPU algorithm (oracle port; sfepy itself is not
installable here) with all host cores on bounded samples of the same workload.
Under torchrun (N > 1) every rank processes its own plates (weak scaling, no collective on the
data path); times are max-over-ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--plates", type=int, default=100)
    ap.add_argument("--conditions", type=int, default=4)
    ap.add_argument("--steps-per-condition", type=int, default=11)
    ap.add_argument("--image-size", type=int, default=64)
    ap.add_argument("--rtol", type=float, default=1e-10)
    ap.add_argument("--max-iter", type=int, default=20000)
    ap.add_argument("--streams", type=int, default=3, help="contexts (streams) the e2e path deals its steps to")
    ap.add_argument("--cpu-samples", type=int, default=32, help="bounded sample for cpu_baseline (about 10 s of CPU work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--distinct-shards", action="store_true", help="every rank draws its own plates for the headline too (N > 1)")
    ap.add_argument("--cpu-mode", default="reference", choices=["reference", "best"],
                    help="--impl reference: re-factorise at every load step like sfepy's ScipyDirect (reference) or "
                         "factor once and scale (best)")
    ap.add_argument("--skip", default="", help="comma list of optional blocks to skip: dataset,as_sampled,c3,c1,cpu_best")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed device-resident step computed as DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


# --------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                pass
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_field(name, key):
    """a field of a committed ncu summary under profiles/ (None if absent)"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", name))).get(key)
    except Exception:
        return None


def ncu_traffic(info, name):
    """dram bytes per launch from the committed ncu capture, if it was taken on this workload."""
    p = os.path.join(ROOT, "profiles", name)
    try:
        t = json.load(open(p))
        if int(t["nnz"]) == int(info["nnz"]) and int(t["n_active_dofs"]) == int(info["n_active_dofs"]):
            return float(t["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


def onchip_roofline(sizes, iters, stats, launch_ms):
    """What bounds k_pcg_cluster: the SM's shared-memory / L1TEX data pipe.  Through it return, per iteration,
    the gathered search-direction entries (16 B per stored 2x2 block), the gather codes (2 B per block), the
    2x2 blocks that live in shared memory or are streamed from L2 (32 B each) and, per block row, 88 B of
    vector traffic (own p and diagonal coupling in the SpMV, p for the iteration's record, p read + written in
    the x/r/p update).  The blocks held in TENSOR MEMORY (tcgen05.ld, 32 B each) use their own datapath and are
    reported beside it.  Block counts per storage tier come from the kernel's own counters (fea_solve_stats),
    peaks from tools/smem_bw.cu and tools/tmem_bw.cu on a B200 of this pool (profiles/*_peak.json)."""
    n_s, nnz_s = sizes
    rows = n_s / 2.0
    rd = {k: float(np.mean([s["cluster_block_reads_" + k] for s in stats])) for k in ("tmem", "smem", "l2")}
    all_reads = rd["tmem"] + rd["smem"] + rd["l2"]
    total = 18.0 * all_reads + 32.0 * (rd["smem"] + rd["l2"]) + float((iters.astype(np.float64) * rows * 88.0).sum())
    peak = ncu_field("smem_peak.json", "stream16_GBs")
    out = {"bound": "shared-memory / L1TEX data pipe", "bytes_per_launch": total,
           "achieved": total / (launch_ms * 1e-3) / 1e9, "unit": "GB/s", "peak": peak,
           "peak_source": "tools/smem_bw.cu on a B200 of this pool (profiles/smem_peak.json): 148 SMs x 126 B/clk",
           "bytes_model": "per iteration: 18 B per stored 2x2 block (16 gathered p + 2 code) + 32 B per block read from shared "
                          "memory or L2 + 88 B per block row; block reads counted by the kernel",
           "block_reads_per_launch": rd,
           "share_of_blocks": {k: (v / all_reads if all_reads else None) for k, v in rd.items()}}
    if peak:
        out["frac"] = out["achieved"] / peak
    tm = None
    try:
        tm = float(json.load(open(os.path.join(ROOT, "profiles", "tmem_peak.json")))["tmem"]["tmem_GBs"])
    except Exception:
        pass
    out["tensor_memory"] = {"bytes_per_launch": 32.0 * rd["tmem"], "achieved": 32.0 * rd["tmem"] / (launch_ms * 1e-3) / 1e9,
                            "unit": "GB/s", "peak": tm, "frac": (32.0 * rd["tmem"] / (launch_ms * 1e-3) / 1e9 / tm) if tm else None,
                            "peak_source": "tools/tmem_bw.cu (profiles/tmem_peak.json): tcgen05.ld.32x32b.x32, 456 B/clk/SM; "
                                           "beside saturating ld.shared traffic both run at 120 B/clk/SM"}
    return out


# --------------------------------------------------------------------------
def oracle_unit(job):
    """One plate-condition through the CPU oracle, reference-faithful: assemble, then factor +
    solve at every loaded step (ScipyDirect without presolve), ranges, the two step-1 images."""
    coors, conn, kw, num_steps, size, affine = job[:6]
    mode = job[6] if len(job) > 6 else "reference"
    from oracle.fea_oracle import OracleProblem
    from oracle import raster_oracle as ro
    p = OracleProblem(coors, conn, num_steps=num_steps, **kw)
    u = p.solve(mode)
    p.ranges_lines(u)
    for c in range(2):
        ro.rasterize_scalar(p.coors, p.conn, u[1][:, c], size, affine)
    return u[-1]


def jobs_of(items, num_steps, mode="reference"):
    return [(it.setup.coors, it.setup.conn, it.kwargs, num_steps, it.size, it.affine, mode) for it in items]


def config_of(a):
    """The workload, in the same words for both arms (the driver compares the two dicts)."""
    return {"workload": workload_name(a), "plates": a.plates, "conditions_per_plate": a.conditions,
            "load_steps": a.steps_per_condition - 1, "mesh_size": 1e-2, "image_size": a.image_size, "seed": a.seed,
            "conditions": "sampler draws kept when well-posed (SURVEY A-19)",
            "l2": "per-step working set (about 400 MB of matrix + 150 MB of vectors) exceeds the 126 MB L2; no flush needed"}


def dist_env():
    from fea_diffusion_b200.sharding import DistEnv
    e = DistEnv.from_env()
    return e.rank, e.world, e.local_rank


def total_of(n, world):
    return n * world


def workload_name(a):
    return ("%d plates x %d conditions x %d load steps, mesh_size 1e-2, image_size %d"
            % (a.plates, a.conditions, a.steps_per_condition - 1, a.image_size))


DUMP_LIMIT = 64 << 20


def dump_outputs(path, res, packed):
    """The BatchResult of one step as path/<name>.npy, so that two builds can be compared output for output on the
    same seeded workload: u (final-step displacement of the kept samples' vertices, concatenated), ranges, iters,
    relres, status and images, in float64 (images in float32), plus sample_index, the plate-conditions kept.  All of
    them are kept while the files stay within DUMP_LIMIT bytes; past that a fixed, seeded sample of them."""
    u = packed.split_vertices(res.u)
    per = np.array([x.nbytes for x in u]) + 4 * res.images[0].size + 8 * 8
    budget = DUMP_LIMIT - 7 * 128    # the .npy headers
    keep = np.arange(packed.n)
    if per.sum() > budget:
        order = np.random.default_rng(0).permutation(packed.n)
        keep = np.sort(order[:np.searchsorted(np.cumsum(per[order]), budget, side="right")])
    arrays = {"sample_index": keep.astype(np.float64), "u": np.concatenate([u[i] for i in keep]),
              "ranges": res.ranges[keep], "iters": res.iters[keep].astype(np.float64), "relres": res.relres[keep],
              "status": res.status[keep].astype(np.float64), "images": res.images[keep].astype(np.float32)}
    os.makedirs(path, exist_ok=True)
    for name, x in arrays.items():
        np.save(os.path.join(path, name + ".npy"), x)


# --------------------------------------------------------------------------
def run_reference(a):
    rank, world, local = dist_env()
    if rank != 0:
        return
    import multiprocessing as mp
    from fea_diffusion_b200.workload import build_workload
    cores = os.cpu_count() or 1
    per_step = 2 * cores
    n_plates = max(1, -(-per_step // a.conditions))
    items, _ = build_workload(n_plates, a.conditions, a.image_size, seed0=a.seed)
    jobs = jobs_of(items[:per_step], a.steps_per_condition, a.cpu_mode)
    with mp.get_context("fork").Pool(cores) as pool:
        for _ in range(a.warmup):
            pool.map(oracle_unit, jobs, chunksize=1)
        t0 = time.perf_counter()
        for _ in range(a.steps):
            pool.map(oracle_unit, jobs, chunksize=1)
        dt = time.perf_counter() - t0
    v = len(jobs) * a.steps / dt
    how = ("re-assembled + scipy SuperLU re-factorised at each of the %d loaded steps (what sfepy's ScipyDirect does)"
           % (a.steps_per_condition - 1)) if a.cpu_mode == "reference" else "factorised once (splu), one solve, load steps scaled (best CPU)"
    sample = "%d plate-conditions per step (first %d plates of the workload), %d worker processes; %s" % (len(jobs), n_plates, cores, how)
    line = {
        "impl": "reference", "metric": "plate-condition FEA solves/sec", "value": v, "unit": "solves/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(a),
        "details": {"note": "CPU oracle = numpy assembly + scipy SuperLU; sfepy itself is not installable here", "cpu_mode": a.cpu_mode},
        "cpu_baseline": {"value": v, "unit": "solves/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------
def run_c3(ctx, a, peak):
    """BASELINE config 3: cantilever L4 / gusset L3 (~1.2-1.3 M DOFs) on the single-GPU streaming path.
    rel-L2 against scipy's sparse LU at the coarse mesh's vertices (tests/golden/c3_lu.npz, made offline by
    tools/make_c3_reference.py: the LU of these systems takes minutes of CPU)."""
    from fea_diffusion_b200 import pack
    from fea_diffusion_b200.workload import large_case
    ref = None
    try:
        ref = np.load(os.path.join(ROOT, "tests", "golden", "c3_lu.npz"))
    except Exception:
        pass
    out = {}
    for name, lv in (("cantilever", 4), ("gusset", 3)):
        setup, n0 = large_case(name, lv)
        packed = pack([setup.sample])
        for rep in range(2):
            with ctx.create_batch(packed) as b:
                ctx.synchronize()
                t0 = time.perf_counter()
                b.assemble()
                ctx.synchronize()
                t1 = time.perf_counter()
                b.solve(1e-10, 400000)
                st, info, r = b.stats(), b.info(), b.download()
        nn, nnz = info["n_active_dofs"], info["nnz"]
        alg = 12 * nnz + 4 * (nn + 1) + 16 * nn
        key = "%s_L%d" % (name, lv)
        e = {"n_dofs": int(nn), "nnz": int(nnz), "iterations": int(st["iterations"]), "status": int(r.status[0]),
             "relres_true": float(r.relres[0]), "assemble_ms": 1e3 * (t1 - t0), "solve_ms": st["solve_ms"],
             "spmv_ms": st["spmv_ms_avg"], "update_ms": st["update_ms_avg"],
             "us_per_iteration": 1e3 * st["solve_ms"] / max(1, st["iterations"]),
             "spmv_algorithmic_GBs": alg / st["spmv_ms_avg"] / 1e6 if st["spmv_ms_avg"] else None,
             "spmv_frac_of_hbm_peak": (alg / st["spmv_ms_avg"] / 1e6 / peak) if st["spmv_ms_avg"] else None,
             "spmv_dram_GBs_ncu": ncu_field("c3_spmv_traffic.json", key)}
        if ref is not None and key + "_u_coarse" in ref:
            g = ref[key + "_u_coarse"]
            e["rel_l2_vs_sparse_lu_at_coarse_vertices"] = float(np.linalg.norm(r.u[:n0] - g) / np.linalg.norm(g))
        out[key] = e
    return out


def run_c1(ctx, a):
    """BASELINE config 1: one plate x one condition x steps_per_condition 5, image 64, through the drop-in
    FEAnalysis (the reference's own per-sample call, generate.py:88-152): latency of the constructor
    (mesh file + region selection), calculate() and the image methods."""
    import shutil
    import tempfile
    from fea_diffusion_b200.datagen import FEAnalysis
    from fea_diffusion_b200.datagen.mesh_generator import write_medit
    from fea_diffusion_b200.workload import plate_conditions
    items, _ = plate_conditions(a.seed, 1, 64)
    it = items[0]
    tmp = tempfile.mkdtemp(prefix="fea_c1_")
    try:
        write_medit(os.path.join(tmp, "part.mesh"), it.setup.coors, it.setup.conn)
        t = {"init_ms": [], "calculate_ms": [], "images_ms": []}
        for rep in range(4):
            cdir = os.path.join(tmp, "1", str(rep))
            os.makedirs(cdir)
            t0 = time.perf_counter()
            an = FEAnalysis("part.mesh", tmp, cdir, num_steps=5, context=ctx, **it.kwargs)
            t1 = time.perf_counter()
            ok = an.calculate()
            t2 = time.perf_counter()
            an.update_image_size_or_bounds(image_size=it.window, bounds=it.bounds)
            an.save_region_images(os.path.join(cdir, "regions"))
            an.save_output_images(os.path.join(cdir, "outputs"), save_stress=False, save_strain=False)
            t3 = time.perf_counter()
            if rep:
                t["init_ms"].append(1e3 * (t1 - t0)); t["calculate_ms"].append(1e3 * (t2 - t1)); t["images_ms"].append(1e3 * (t3 - t2))
        return {"workload": "1 plate x 1 condition x 5 steps, image 64 (seed %d, %d vertices)" % (a.seed, len(it.setup.coors)),
                "ok": bool(ok), "iterations": int(an.iterations),
                "init_ms": float(np.median(t["init_ms"])), "calculate_ms": float(np.median(t["calculate_ms"])),
                "images_ms": float(np.median(t["images_ms"])),
                "note": "calculate() = the reference's own TIME: bracket (generate.py:109-111); it includes writing domain.k.vtk + regions.vtk"}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


# --------------------------------------------------------------------------
def run_b200(a):
    rank, world, local = dist_env()
    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        torch.cuda.set_device(local)
        # NCCL is registered for CUDA tensors, gloo for CPU tensors.  The data path has no collective;
        # the barrier and the max-over-ranks of the timings are host scalars and go over gloo unless
        # FEA_BENCH_NCCL=1 (an initialised NCCL communicator was measured to slow the persistent
        # cluster kernels by ~8 %, so it is only created when asked for)
        dist.init_process_group("cpu:gloo,cuda:nccl")
    use_nccl = os.environ.get("FEA_BENCH_NCCL", "0") == "1"
    # the library __graft_entry__.build() left in the tree; the bench compiles nothing and writes nothing there
    from fea_diffusion_b200 import Context, load_library, pack
    load_library()
    from fea_diffusion_b200.solver import BatchResult
    from fea_diffusion_b200.workload import build_workload

    t_gen = time.perf_counter()
    from fea_diffusion_b200.sharding import reduce_scalar, weak_scaling_seed
    # weak scaling: every rank solves the SAME synthetic workload (same plate seeds), so the per-GPU
    # work is identical by construction and the N-GPU figure measures the machine, not the draw of
    # plates (two 100-plate draws differ by +-15 % in PCG work); --distinct-shards gives every rank
    # its own plates instead
    seed0 = weak_scaling_seed(a.seed, rank) if a.distinct_shards else a.seed
    cache = os.environ.get("FEA_BENCH_CACHE")   # tuning sessions: reuse the generated workload between runs
    if cache:
        import pickle
        cache = "%s.%d.%d.%d.%d.pkl" % (cache, a.plates, a.conditions, a.image_size, seed0)
    skip = set(x for x in a.skip.split(",") if x)
    # N > 1 without --distinct-shards: every rank solves the SAME workload, so rank 0 alone generates it (all
    # cores) and hands it over through a file on the node; the other ranks meanwhile generate the plates of
    # their own dataset_e2e shard (8 ranks x all-core pools on one box would oversubscribe the host 8x)
    share = None
    if world > 1 and not a.distinct_shards and not cache:
        import pickle
        share = os.path.join(os.environ.get("TMPDIR", "/tmp"), "fea_bench_workload.%s.%s.pkl"
                             % (os.environ.get("MASTER_PORT", "0"), os.environ.get("TORCHELASTIC_RUN_ID", "run")))
    ds_items = None
    if share and rank > 0:
        if "dataset" not in skip:
            ds_items, _ = build_workload(a.plates, a.conditions, a.image_size, seed0=weak_scaling_seed(a.seed, rank),
                                         workers=max(1, (os.cpu_count() or 1) // world))
        dist.all_reduce(torch.zeros(1))   # host barrier over gloo (CPU tensor): rank 0 has written the file
        with open(share, "rb") as f:
            items, rejected, extras = pickle.load(f)
        dist.all_reduce(torch.zeros(1))   # everybody has read it: rank 0 removes it
    elif cache and os.path.exists(cache):
        with open(cache, "rb") as f:
            items, rejected, extras = pickle.load(f)
    else:
        items, rejected, extras = build_workload(a.plates, a.conditions, a.image_size, seed0=seed0,
                                                 extra_as_sampled=a.conditions, workers=os.cpu_count() or 1)
        if cache and rank == 0:
            with open(cache, "wb") as f:
                pickle.dump((items, rejected, extras), f)
        if share:
            with open(share + ".tmp", "wb") as f:
                pickle.dump((items, rejected, extras), f)
            os.replace(share + ".tmp", share)
            dist.all_reduce(torch.zeros(1))
            dist.all_reduce(torch.zeros(1))
            os.remove(share)
    # dataset_e2e at N > 1: every rank synthesises its OWN plates (the dataset is sharded, not replicated)
    if ds_items is None:
        ds_items = items
    t_gen = time.perf_counter() - t_gen
    n = len(items)
    ctx = Context(local)
    packed = pack([it.setup.sample for it in items], alloc=ctx.pinned_empty)
    size = max(it.size for it in items)
    affine = np.stack([it.affine for it in items])
    t1 = float(np.linspace(0.0, 1.0, a.steps_per_condition)[1])

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        if dist is not None:
            if use_nccl:
                dist.barrier(device_ids=[local])
                torch.cuda.synchronize()   # the NCCL barrier kernel spins on SMs until the peers arrive: wait it out
            else:
                t = torch.zeros(1)
                dist.all_reduce(t)         # gloo: a host-side barrier

    def max_over_ranks(x):
        return reduce_scalar(x, "max", device="cuda" if (dist is not None and use_nccl) else None)

    def device_step(batch):
        batch.assemble().solve(a.rtol, a.max_iter).rasterize(size, affine, t1)

    # ---- device-resident throughput: inputs uploaded before the timed region; one stream, so the
    # per-launch CUDA events around the SpMV see that kernel alone ---------------------------------
    for w in range(max(a.warmup, 1)):
        # same shape as the timed loop (a.steps batches alive at once) so the stream-ordered
        # memory pool has its final size before timing starts
        wb = [ctx.create_batch(packed) for _ in range(a.steps)] if w == 0 else [ctx.create_batch(packed)]
        for b in wb:
            device_step(b)
        for b in wb:
            b.destroy()
    batches = [ctx.create_batch(packed) for _ in range(a.steps)]
    clocks = ClockSampler(local)
    clocks.start()
    launches0 = ctx.kernel_launches()
    barrier()
    ctx.event_record(0)
    for b in batches:
        device_step(b)
    ctx.event_record(1)
    barrier()
    ms_dev = max_over_ranks(ctx.event_elapsed_ms(0, 1))
    launches = ctx.kernel_launches() - launches0
    info = batches[0].info()
    sizes = batches[0].sample_sizes()
    stats = [b.stats() for b in batches]
    cl_size = stats[0]["cluster_size"]
    res0 = batches[0].download()
    rounds0 = batches[0].refine_rounds()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, batches[-1].download(images=True), packed)
    for b in batches:
        b.destroy()

    # ---- end to end through the public host-buffer API: every step copies its inputs from pinned
    # host memory and reads u, ranges, images back.  Steps are dealt to a.streams contexts (one
    # stream + one host thread each) so that copies, host polls and the low-occupancy tail of one
    # batch overlap the bulk of another (fea_diffusion_b200.pipeline.Pipeline) ---------------------
    from fea_diffusion_b200.pipeline import Pipeline
    a.streams = max(1, min(a.streams, a.steps // 2))   # at least two steps per stream, or there is nothing to overlap
    # the pipeline's host threads hand the GIL to each other between ctypes calls: with the default 5 ms
    # switch interval a thread that packs the next batch (pure Python + numpy) stalls the launch chain of the others
    sys.setswitchinterval(float(os.environ.get("FEA_BENCH_SWITCH_INTERVAL", "0.001")))
    pipe = Pipeline(local, a.streams, staggered_priorities=False, first=ctx)
    outs = [BatchResult(u=c.pinned_empty((packed.n_vertices, 2), np.float64), ranges=c.pinned_empty((n, 4), np.float64),
                        iters=c.pinned_empty((n,), np.int32), relres=c.pinned_empty((n,), np.float64),
                        status=c.pinned_empty((n,), np.int32), images=c.pinned_empty((n, 2, size, size), np.uint8))
            for c in pipe.ctxs]

    def e2e_step(c, j):
        c.solve_batch(packed, a.rtol, a.max_iter, size, affine, t1, out=outs[pipe.ctxs.index(c)])

    pipe.run(list(range(max(a.warmup, a.streams))), e2e_step)
    pipe.synchronize()
    barrier()
    ctx.event_record(2)
    pipe.run(list(range(a.steps)), e2e_step)
    pipe.join_into(ctx)
    ctx.event_record(3)
    barrier()
    ms_e2e = max_over_ranks(ctx.event_elapsed_ms(2, 3))
    clk = clocks.stop()
    out = outs[0]
    h2d = packed.h2d_bytes + affine.nbytes
    d2h = out.u.nbytes + out.ranges.nbytes + out.iters.nbytes + out.relres.nbytes + out.status.nbytes + out.images.nbytes
    e2e_ok = all(np.array_equal(o.status, res0.status) and np.array_equal(o.u, res0.u) for o in outs[:min(a.streams, a.steps)])

    # ---- dataset end to end: in-memory meshes + condition dicts -> u, ranges, images, region images.
    # Timed region per step: host packing of the condition dicts into flat (pinned) arrays, H2D,
    # region selection / Dirichlet mask / material cells / load on the device, assemble, solve, raster
    # of the displacement and of every region (+ the plate mask of input.png), the A-19 classifier,
    # D2H of everything a writer needs.  Outside: meshing, the condition sampler, PNG / text encoding.
    from fea_diffusion_b200.solver import PackedConditions, PinnedArena
    from fea_diffusion_b200.workload import conditions_of
    dataset = None
    if "dataset" not in skip:
        ds_meshes, ds_samples = conditions_of(ds_items)
        ds_size = max(it.size for it in ds_items)
        ds_affine = np.stack([it.affine for it in ds_items])
        ds_mask = np.array([it.condition == 0 for it in ds_items], np.uint8)
        probe = PackedConditions(ds_meshes, ds_samples)
        n_img = int(probe.n_regions.sum() + ds_mask.sum())
        # Three host threads on one GPU: a packer turns the condition dicts of step j + 1 into flat pinned arrays and
        # uploads the big ones (coordinates, connectivity, material coordinate lists) on a context of its own; the
        # compute thread drives step j on the main context (create -> assemble -> solve -> rasters -> region rasters +
        # classifier staged on the device, fea_batch_stage_outputs); a reader fetches step j - 1 on a second context's
        # stream (fea_batch_fetch_outputs), so the ~60 MB of D2H copies run on a copy engine under the next solve.
        # (Dealing whole steps to several contexts, as the e2e path does, serialises here: the small kernels of one
        # context's step cannot run while another context's solve has CTAs pending, so every synchronising call of a
        # step waits for a foreign solve -- measured 55.6 ms per step with 3 contexts, 51 with 2, 38.4 with one
        # context doing everything in turn.)
        import queue
        copy_ctx, up_ctx = Context(local), Context(local)
        arenas = [PinnedArena(ctx, probe.h2d_bytes + (1 << 20)) for _ in range(4)]
        ds_outs = [BatchResult(u=ctx.pinned_empty((probe.n_vertices, 2), np.float64), ranges=ctx.pinned_empty((n, 4), np.float64),
                               iters=ctx.pinned_empty((n,), np.int32), relres=ctx.pinned_empty((n,), np.float64),
                               status=ctx.pinned_empty((n,), np.int32), images=ctx.pinned_empty((n, 2, ds_size, ds_size), np.uint8))
                   for _ in range(2)]
        ds_regs = [ctx.pinned_empty((n_img, ds_size, ds_size), np.uint8) for _ in range(2)]
        ds_cls = [None]
        pack_s, phase_s, fetch_s, upload_s, errs = [], [], [], [], []

        def run_dataset(n_steps):
            q, dq, done = queue.Queue(maxsize=1), queue.Queue(maxsize=1), queue.Queue()

            go = threading.Semaphore(1)   # the packer (pure Python + numpy: it holds the GIL) works while the compute
                                          # thread sits in the solve call (GIL released), not beside its launch chain

            def packer():
                for j in range(n_steps):
                    go.acquire()
                    t0 = time.perf_counter()
                    ar = arenas[j % 4]        # in flight at most: one being read back, one consumed, one queued, one being packed
                    ar.reset()
                    pc = PackedConditions(ds_meshes, ds_samples, alloc=ar.empty)
                    pack_s.append(time.perf_counter() - t0)
                    t0 = time.perf_counter()
                    ar.upload(up_ctx)         # H2D of the big arrays on the packer's own context, under the running solve
                    pc.use_device_copy(ar)
                    upload_s.append(time.perf_counter() - t0)
                    q.put(pc)

            def reader():
                for j in range(n_steps):
                    b = dq.get()
                    t0 = time.perf_counter()
                    try:
                        _, _, ds_cls[0] = b.fetch_outputs(copy_ctx, out=ds_outs[j % 2], regions=ds_regs[j % 2])
                    except Exception as e:    # keep draining so that the compute thread never blocks on a dead reader
                        errs.append(e)
                    fetch_s.append(time.perf_counter() - t0)
                    done.put(b)           # destroyed by the compute thread (its context frees the device memory)

            ths = [threading.Thread(target=packer), threading.Thread(target=reader)]
            for th in ths:
                th.start()
            for j in range(n_steps):
                t0 = time.perf_counter()
                pc = q.get()
                t1_ = time.perf_counter()
                while not done.empty():
                    done.get().destroy()
                b = ctx.create_batch_from_conditions(pc)
                t2_ = time.perf_counter()
                b.assemble()
                go.release()
                b.solve(a.rtol, a.max_iter).rasterize(ds_size, ds_affine, t1).stage_outputs(ds_mask)
                t3_ = time.perf_counter()
                dq.put(b)
                phase_s.append((t1_ - t0, t2_ - t1_, t3_ - t2_, time.perf_counter() - t3_))
            for th in ths:
                th.join()
            while not done.empty():
                done.get().destroy()
            if errs:
                raise errs[0]
            return (n_steps - 1) % 2

        pipe.synchronize()
        run_dataset(max(a.warmup, 2))
        ctx.synchronize()
        pack_s.clear()
        phase_s.clear()
        fetch_s.clear()
        upload_s.clear()
        barrier()
        ctx.event_record(4)
        t0 = time.perf_counter()
        n_ds = a.steps               # the pipeline's fill (packing step 0) and drain (last read-back) are inside the timed region
        last = run_dataset(n_ds)
        ctx.event_record(5)
        barrier()
        wall_ms = 1e3 * (time.perf_counter() - t0)
        ms_ds = max_over_ranks(max(ctx.event_elapsed_ms(4, 5), wall_ms))
        copy_ctx.synchronize()
        o = ds_outs[last]
        fl, em = ds_cls[0]
        same = (ds_items is items and np.array_equal(o.status, res0.status) and np.array_equal(o.u, res0.u))
        dataset = {"value": total_of(n, world) * n_ds / (ms_ds * 1e-3), "unit": "samples/s", "ms_per_step": ms_ds / n_ds, "steps": n_ds,
                   "h2d_bytes_per_step": int(probe.h2d_bytes + ds_affine.nbytes + ds_mask.nbytes),
                   "d2h_bytes_per_step": int(o.u.nbytes + o.ranges.nbytes + o.iters.nbytes + o.relres.nbytes + o.status.nbytes
                                             + o.images.nbytes + ds_regs[0].nbytes + 8 * n),
                   "host_pack_ms_per_step": 1e3 * float(np.mean(pack_s)) if pack_s else None,
                   "compute_thread_ms_per_step": dict(zip(("wait_for_packer", "create_from_conditions",
                                                           "assemble_solve_raster_stage_regions_classifier", "hand_over"),
                                                          (1e3 * np.mean(phase_s, axis=0)).round(2).tolist())) if phase_s else None,
                   "reader_thread_fetch_ms_per_step": round(1e3 * float(np.mean(fetch_s)), 2) if fetch_s else None,
                   "packer_thread_upload_ms_per_step": round(1e3 * float(np.mean(upload_s)), 2) if upload_s else None,
                   "host_threads": "packer thread (packs step j + 1 and uploads its big arrays on a context of its own) + compute "
                                   "thread (main context) + reader thread (copy context: D2H of step j - 1), all under the solve of step j",
                   "timer": "max(wall clock until the last read-back has returned, CUDA events) around %d steps, max over ranks" % n_ds,
                   "region_images_per_step": n_img, "pinned_arena_spills": int(sum(x.spilled for x in arenas)),
                   "classifier": {"well_posed": int(((fl == 0) & (em == 0)).sum()), "floating": int((fl > 0).sum()),
                                  "empty_rows": int((em > 0).sum())},
                   "shards": ("every rank synthesises its own plates (rank r: seeds %d + 100000 r ...)" % a.seed) if world > 1
                             else "one shard",
                   "bytes_identical_to_device_resident_run": bool(same) if ds_items is items else None,
                   "includes": "host packing of condition dicts, H2D, device region selection + Dirichlet mask + load "
                               "(fea_batch_create_from_conditions), assemble, solve, displacement + region rasters, "
                               "A-19 classifier, D2H",
                   "excludes": "meshing, condition sampler, PNG/text encoding (north_star: host, outside the timed path)"}

    # ---- as sampled: the sampler's own condition distribution (reference mesh_generator.py:397-521; a
    # third of the draws singular by construction, SURVEY F4) through the same device path ----------
    as_sampled = None
    if "as_sampled" not in skip and extras:
        plate_of = {}
        for it in items:
            plate_of.setdefault(it.plate, (it.setup.coors, it.setup.conn))
        as_meshes = list(plate_of.values())
        as_samples = [(i, kw) for i, ex in enumerate(extras) for kw in ex]
        pc = PackedConditions(as_meshes, as_samples)
        as_aff = np.stack([items[i * a.conditions].affine for i, ex in enumerate(extras) for _ in ex])
        for rep in range(2):
            ctx.synchronize()
            ctx.event_record(6)
            with ctx.create_batch_from_conditions(pc) as b:
                b.assemble().solve(a.rtol, a.max_iter).rasterize(size, as_aff, t1)
                ctx.event_record(7)
                r_as = b.download()
                fl, em = b.classify()
            ms_as = ctx.event_elapsed_ms(6, 7)
        names = {0: "converged", 1: "max_iter", 2: "breakdown", 3: "empty_row", 4: "stagnated"}
        hist = {names[k]: int((r_as.status == k).sum()) for k in names}
        wp = (fl == 0) & (em == 0)
        as_sampled = {"samples": len(as_samples), "ms_per_batch": ms_as, "samples_per_s": len(as_samples) / (ms_as * 1e-3),
                      "status": hist,
                      "classifier": {"well_posed": int(wp.sum()), "floating_parts": int((fl > 0).sum()), "empty_rows": int((em > 0).sum())},
                      "well_posed_not_converged": int((wp & (r_as.status != 0)).sum()),
                      "ill_posed_reported_converged": int((~wp & (r_as.status == 0)).sum()),
                      "note": "conditions exactly as the sampler draws them, material regions by the reference's own methods "
                              "(KMeans over flattened centres / agglomerative, scikit-learn); the reference writes SuperLU noise "
                              "for the singular ones"}

    # ---- roofline of the dominant kernel --------------------------------------------------------
    # Plate-sized systems are solved on chip (k_pcg_cluster: one system per thread-block cluster,
    # matrix in shared memory): ONE launch per step whose algorithmic bytes are the PCG iterations
    # it performs, sum_s iters_s * B_iter(s) with SURVEY 8(d)'s B_iter = 12 nnz + 4 (n+1) + 8 n + 96 n.
    # Systems too large for a cluster use the streaming kernels; then the SpMV launch is reported.
    peak, peak_src = measured_peak()
    nn, nnz = info["n_active_dofs"], info["nnz"]
    on_chip = sum(s["cluster_systems"] for s in stats) > 0
    if on_chip:
        n_s, nnz_s = sizes
        b_iter = 12.0 * nnz_s + 4.0 * (n_s + 1) + 8.0 * n_s + 96.0 * n_s
        alg_bytes = float((res0.iters.astype(np.float64) * b_iter).sum())
        ms = float(np.mean([s["cluster_ms"] for s in stats]))
        achieved = alg_bytes / (ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "k_pcg_cluster<1..8> (one persistent kernel per cluster size, launched "
                                              "concurrently; most systems ran on %d-CTA clusters)" % cl_size,
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "frac_note": "algorithmic bytes vs the HBM peak, ON-CHIP regime: > 1 by design (the matrix crosses HBM once "
                                 "per solve, not once per iteration); the resource that bounds the kernel is in 'onchip'",
                    "traffic": ncu_traffic(info, "cluster_traffic.json"), "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": ms,
                    "timed_launches": len(stats), "pcg_iterations_in_launch": int(res0.iters.sum()),
                    "regime": "on-chip: each system's matrix is read from HBM once per solve into the tensor memory and shared "
                              "memory of a thread-block cluster and its CG vectors stay in registers, so achieved algorithmic GB/s "
                              "exceeds the HBM peak by design; HBM-streaming figures of the same iterations are in "
                              "'streaming_path'",
                    "clusters": stats[0]["cluster_count"], "systems_on_chip": stats[0]["cluster_systems"],
                    "onchip": onchip_roofline(sizes, res0.iters, stats, ms),
                    "onchip_pipe": ncu_field("cluster_traffic.json", "onchip_pipe"),
                    "l2_read_peak_gbs": 17900.0, "hbm_read_peak_gbs": 6880.0,
                    "peaks_note": "L2-resident / HBM-resident read bandwidth measured with tools/l2_bw.cu on a B200 of this pool"}
    else:
        roofline = None
    # the streaming kernels on the same batch (one extra, untimed-region solve): the HBM-bound SpMV
    ctx.set_option("pcg_path", 1)
    with ctx.create_batch(packed) as sb:
        sb.assemble().solve(a.rtol, a.max_iter)
        sst = sb.stats()
    ctx.set_option("pcg_path", 0)
    spmv_bytes = 12 * nnz + 4 * (nn + n) + 16 * nn            # SURVEY 8(d): B_spmv, s = 1
    moved = 36 * info["sell_blocks"] + 4 * (info["block_rows"] // 32) * 3 + 16 * info["block_rows"] * 4
    streaming = {"kernel": "k_pcg_spmv", "achieved": spmv_bytes / (sst["spmv_ms_avg"] * 1e-3) / 1e9 if sst["spmv_ms_avg"] else None,
                 "peak": peak, "unit": "GB/s", "algorithmic_bytes_per_launch": spmv_bytes, "layout_bytes_per_launch": moved,
                 "launch_ms": sst["spmv_ms_avg"], "update_kernel_ms": sst["update_ms_avg"], "solve_ms": sst["solve_ms"],
                 "timed_launches": sst["spmv_launches_timed"], "traffic": ncu_traffic(info, "spmv_traffic.json")}
    if streaming["achieved"]:
        streaming["frac"] = streaming["achieved"] / peak
    if roofline is None:
        roofline = dict(streaming, bound="hbm", peak_source=peak_src)
    else:
        roofline["streaming_path"] = streaming

    total = total_of(n, world)
    line = {
        "metric": "plate-condition FEA solves/sec", "value": total * a.steps / (ms_dev * 1e-3), "unit": "solves/s",
        "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_dev / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(a),
        "details": {"samples_per_gpu": n, "active_dofs_per_gpu": nn, "nnz_per_gpu": nnz,
                    "rtol": a.rtol, "pcg_iterations_max": int(res0.iters.max()), "pcg_iterations_mean": float(res0.iters.mean()),
                    "converged": int((res0.status == 0).sum()),
                    "stagnated_ill_conditioned": int((res0.status == 4).sum()), "refined_in_extended_precision": int(stats[0]["refined_systems"]),
                    "sell_padding": info["sell_blocks"] * 4.0 / max(1, nnz),
                    "matrix_bytes_per_step": int(36 * info["sell_blocks"]),
                    "solver_path": "on-chip cluster PCG" if on_chip else "streaming PCG",
                    "conditions_rejected_as_ill_posed": rejected, "input_generation_s": round(t_gen, 1),
                    "parallelism": "samples sharded per GPU, no collective; %s"
                                   % ("every rank has its own plates" if a.distinct_shards else
                                      "value / e2e: every rank solves the same 100-plate workload (identical per-GPU work); "
                                      "dataset_e2e: every rank has its own plates")},
        "e2e": {"value": total * a.steps / (ms_e2e * 1e-3), "unit": "solves/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e / a.steps, "streams": a.streams,
                "bytes_identical_to_device_resident_run": bool(e2e_ok)},
        "gpu_launches": int(launches), "clocks": clk, "roofline": roofline,
        "dataset_e2e": dataset, "as_sampled": as_sampled,
    }
    if rank == 0 and world == 1:
        if "c3" not in skip:
            line["c3"] = run_c3(ctx, a, peak)
        if "c1" not in skip:
            line["c1"] = run_c1(ctx, a)
    # ---- CPU baseline beside it (rank 0, N = 1 only) ------------------------------------------
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        jobs = jobs_of(items[:a.cpu_samples], a.steps_per_condition)
        t0 = time.perf_counter()
        u_cpu = [oracle_unit(j) for j in jobs]
        dt = time.perf_counter() - t0
        # the same samples from the timed GPU step against the CPU direct solve (north_star: <= 1e-8)
        u_gpu = packed.split_vertices(res0.u)
        # samples the solver does NOT report as converged (FEAnalysis.calculate() returns False for them and the
        # generator redraws the condition) are listed, not compared: there is no converged result to compare
        conv = [i for i in range(len(jobs)) if int(res0.status[i]) == 0]
        rel = lambda i: float(np.linalg.norm(u_gpu[i] - u_cpu[i]) / np.linalg.norm(u_cpu[i]))
        plain = [i for i in conv if rounds0[i] == 0]
        errs = [rel(i) for i in plain]
        not_conv = {int(i): rel(i) for i in range(len(jobs)) if i not in conv and np.isfinite(u_gpu[i]).all()}
        # samples the solver flags as ill-conditioned (fp64 CG stalled above the tolerance; finished with
        # double-double residual rounds): the direct solve's own answer is only defined to ~kappa eps there.
        # Listed with the band by which SuperLU's solution moves when K is perturbed by half an ulp.
        from oracle.fea_oracle import OracleProblem
        from oracle.sensitivity import direct_solve_sensitivity
        flagged = {}
        for i in conv:
            if rounds0[i] > 0:
                it = items[i]
                orc = OracleProblem(it.setup.coors, it.setup.conn, num_steps=2, **it.kwargs)
                band = direct_solve_sensitivity(orc.stiffness(), orc.rhs_final())
                e_best = float(np.linalg.norm(u_gpu[i] - orc.solve("best")[-1]) / np.linalg.norm(u_cpu[i]))
                flagged[int(i)] = {"rel_l2_vs_cpu_direct_solve": e_best, "rel_l2_vs_cpu_reference_mode_10_refactorisations": rel(i),
                                   "cpu_direct_solve_moves_by_when_K_is_perturbed_half_an_ulp": band,
                                   "refinement_rounds": int(rounds0[i]), "true_relres": float(res0.relres[i]),
                                   "within_band": bool(e_best <= 1e-8 + 4.0 * band)}
        line["parity"] = {"samples": len(plain), "max_rel_l2_vs_cpu_direct_solve": max(errs) if errs else None, "tolerance": 1e-8,
                          "ok": bool(errs and max(errs) <= 1e-8 and not not_conv and all(v["within_band"] for v in flagged.values())),
                          "flagged_ill_conditioned": {"count": len(flagged), "samples": flagged,
                                                      "rule": "rel-L2 <= 1e-8 + 4 x the direct solve's own half-ulp band"},
                          "reported_not_converged": {"count": len(jobs) - len(conv), "rel_l2_vs_cpu_direct_solve": not_conv},
                          "images_note": "images are checked in tests/ (bit-exact to the raster oracle for the same u, within 1 LSB end "
                                         "to end); that oracle is pinned to VTK's committed renders on INTERIOR pixels only -- VTK's "
                                         "edge-pixel coverage rule is not recoverable without VTK (SURVEY A-16)"}
        line["cpu_baseline"] = {"value": len(jobs) / dt, "unit": "solves/s", "cores": 1, "kind": "port",
                                "host_cores_available": os.cpu_count(),
                                "sample": "first %d plate-conditions of the workload, %.1f s, reference-faithful "
                                          "(SuperLU re-factorised at each load step)" % (len(jobs), dt)}
        if "cpu_best" not in skip:
            # best CPU: factor once (splu), one solve, load steps scaled -- what the GPU path itself exploits (F5)
            jb = jobs_of(items[:a.cpu_samples], a.steps_per_condition, "best")
            t0 = time.perf_counter()
            for j in jb:
                oracle_unit(j)
            dtb = time.perf_counter() - t0
            best = {"value": len(jb) / dtb, "unit": "solves/s", "cores": 1, "kind": "port",
                    "sample": "first %d plate-conditions, %.1f s, factorised once + scaled load steps" % (len(jb), dtb)}
            try:   # all cores: the reference arm of this script in its own process (no CUDA context in the workers)
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--cpu-mode", "best",
                                    "--steps", "2", "--warmup", "1", "--conditions", str(a.conditions), "--image-size", str(a.image_size),
                                    "--steps-per-condition", str(a.steps_per_condition), "--seed", str(a.seed)],
                                   capture_output=True, text=True, timeout=600)
                jl = json.loads(r.stdout.strip().splitlines()[-1])
                best["all_cores"] = {"value": jl["value"], "cores": jl["cpu_baseline"]["cores"], "sample": jl["cpu_baseline"]["sample"]}
            except Exception as e:   # report, never fail the bench on the side measurement
                best["all_cores"] = {"error": repr(e)[:200]}
            line["cpu_baseline_best"] = best
            line["vs_best_cpu"] = {"e2e_over_1_core": line["e2e"]["value"] / best["value"],
                                   "e2e_over_all_cores": (line["e2e"]["value"] / best["all_cores"]["value"])
                                   if "value" in best["all_cores"] else None}
    if rank == 0:
        print(json.dumps(line), flush=True)
    pipe.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
