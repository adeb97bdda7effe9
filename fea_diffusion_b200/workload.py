"""Synthetic workloads for bench.py and the large-solve tests: BASELINE.json's configurations
built from the seeded plate generator (SURVEY.md section 8d)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Tuple

import numpy as np

from . import imaging
from .host import MeshTopology, ProblemSetup, floating_components
from .plates import condition_kwargs, make_plate


@dataclass
class WorkItem:
    plate: int
    condition: int
    setup: ProblemSetup
    kwargs: Dict                 # FEAnalysis-style arguments (for the CPU oracle)
    window: int                  # modified_image_size of the plate
    bounds: Tuple[int, int, int, int]
    affine: np.ndarray           # world -> crop pixel
    size: int                    # crop size (pixels)


def plate_conditions(seed: int, conditions_per_plate: int, image_size: int, mesh_size: float = 1e-2,
                     well_posed: bool = True, max_draws: int = 400, extra_as_sampled: int = 0,
                     as_sampled_method: str = "reference"):
    """All conditions of one plate.  With ``well_posed`` the condition sampler is redrawn until
    every stiffness-connected component carries >= 2 fixed vertices and no active vertex is
    isolated (SURVEY A-19); the number of rejected draws is returned for the report."""
    gen, ptags, ltags = make_plate(seed, mesh_size)
    coors, conn = gen.mesh
    topo = MeshTopology(conn, len(coors))
    bbox = (float(coors[:, 0].min()), float(coors[:, 1].min()), float(coors[:, 0].max()), float(coors[:, 1].max()))
    window, bounds = imaging.plate_window(bbox, image_size)
    affine = imaging.crop_affine(bbox, window, bounds)
    items: List[WorkItem] = []
    rejected = 0
    draws = 0
    while len(items) < conditions_per_plate:
        if draws >= max_draws:
            raise RuntimeError("plate %d: no well-posed condition in %d draws" % (seed, max_draws))
        cond = gen.sample_conditions(ptags, ltags, 1)[0]
        draws += 1
        kw = condition_kwargs(cond)
        setup = ProblemSetup(coors, conn, topology=topo, **kw)
        if well_posed and floating_components(setup.sample) != (0, 0):
            rejected += 1
            continue
        items.append(WorkItem(seed, len(items), setup, kw, window, bounds, affine, bounds[2] - bounds[0]))
    if extra_as_sampled:
        # further draws of the same plate exactly as the sampler produces them (the reference's own
        # distribution, a third of it singular by construction, SURVEY F4): condition dicts only,
        # the device derives everything else (fea_batch_create_from_conditions)
        # -- with the reference's own region methods (KMeans / agglomerative, plates.py) on the same mesh,
        # from a sampler stream of their own
        import copy
        import random
        g2 = copy.copy(gen)
        g2.region_method = as_sampled_method
        g2.random = random.Random(seed * 7919 + 17)
        extra = [condition_kwargs(c) for c in g2.sample_conditions(ptags, ltags, extra_as_sampled)]
        return items, rejected, extra
    return items, rejected


def _plate_job(a):
    try:   # one thread per worker process: the pool already uses every core (scikit-learn / BLAS would each take all)
        from threadpoolctl import threadpool_limits
        with threadpool_limits(1):
            return plate_conditions(a[0], a[1], a[2], a[3], a[4], extra_as_sampled=a[5])
    except ImportError:
        return plate_conditions(a[0], a[1], a[2], a[3], a[4], extra_as_sampled=a[5])


def build_workload(n_plates: int, conditions_per_plate: int = 4, image_size: int = 64, seed0: int = 0,
                   mesh_size: float = 1e-2, well_posed: bool = True, extra_as_sampled: int = 0, workers: int = 1):
    """(items, rejected draws[, as-sampled condition kwargs per plate]).  Plates are independent and seeded
    one by one, so ``workers`` > 1 (a fork pool: call it before the process owns a CUDA context) returns the
    same workload as the serial loop."""
    items: List[WorkItem] = []
    rejected = 0
    extras = []
    jobs = [(seed0 + p, conditions_per_plate, image_size, mesh_size, well_posed, extra_as_sampled) for p in range(n_plates)]
    if workers > 1 and n_plates > 1:
        import multiprocessing as mp
        if extra_as_sampled:
            try:   # imported once here, inherited by the forked workers (seconds per process otherwise)
                import sklearn.cluster  # noqa: F401
            except ImportError:
                pass
        with mp.get_context("fork").Pool(min(workers, n_plates)) as pool:
            results = pool.map(_plate_job, jobs, chunksize=1)
    else:
        results = [_plate_job(j) for j in jobs]
    for r in results:
        items.extend(r[0])
        rejected += r[1]
        if extra_as_sampled:
            extras.append(r[2])
    if extra_as_sampled:
        return items, rejected, extras
    return items, rejected


def conditions_of(items: List[WorkItem]):
    """(meshes, samples) for ``solver.PackedConditions``: the distinct plate meshes of ``items`` and
    one (mesh index, FEAnalysis kwargs) pair per item -- the in-memory form of what the reference's
    generate loop hands to FEAnalysis (generate.py:88-107)."""
    meshes, samples, index = [], [], {}
    for it in items:
        if it.plate not in index:
            index[it.plate] = len(meshes)
            meshes.append((it.setup.coors, it.setup.conn))
        samples.append((index[it.plate], it.kwargs))
    return meshes, samples


def refine_uniform(coors: np.ndarray, conn: np.ndarray, levels: int):
    """Uniform red refinement (each triangle -> 4; midpoints appended after the existing
    vertices), the mesh family of BASELINE config 3 (SURVEY C-5; the reference's
    ``refine_mesh`` hook, applications/cantilever/cantilever.py:26-27)."""
    coors = np.asarray(coors, dtype=np.float64)
    conn = np.asarray(conn, dtype=np.int64)
    for _ in range(levels):
        n = len(coors)
        e = np.concatenate([conn[:, [0, 1]], conn[:, [1, 2]], conn[:, [2, 0]]])
        key = np.minimum(e[:, 0], e[:, 1]) * n + np.maximum(e[:, 0], e[:, 1])
        uniq, inv = np.unique(key, return_inverse=True)
        mid = 0.5 * (coors[uniq // n] + coors[uniq % n])
        m = (n + inv).reshape(3, -1).T  # midpoints of edges (01, 12, 20) per cell
        a, b, c = conn[:, 0], conn[:, 1], conn[:, 2]
        ab, bc, ca = m[:, 0], m[:, 1], m[:, 2]
        conn = np.concatenate([np.stack([a, ab, ca], 1), np.stack([ab, b, bc], 1),
                               np.stack([ca, bc, c], 1), np.stack([ab, bc, ca], 1)])
        coors = np.concatenate([coors, mid])
    return np.ascontiguousarray(coors), np.ascontiguousarray(conn.astype(np.int32))


def large_case(name: str, levels: int, fixtures_path: str = None):
    """BASELINE config 3: the reference's cantilever / gusset application problems
    (applications/cantilever/cantilever.py:43-52, applications/gusset/gusset.py:39-94) on their
    meshes refined ``levels`` times (the ``refine_mesh`` hook, cantilever.py:26-27).  Returns
    (ProblemSetup, n_coarse_vertices): the coarse mesh's vertices keep their indices under refinement."""
    import os
    if fixtures_path is None:
        fixtures_path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "fixtures.npz")
    F = np.load(fixtures_path)
    c0, n0 = F[name + "_coors"], F[name + "_conn"]
    co, cn = refine_uniform(c0, n0, levels)
    setup = ProblemSetup(co, cn)
    topo = MeshTopology(setup.conn, len(co))
    from .host import vertices_on_line
    if name == "cantilever":
        fixed = topo.facet_vertices(np.flatnonzero(co[:, 0] < 0.01))
        loads = [(np.array([3]), (0.0, -1000.0))]
    elif name == "gusset":
        fixed = topo.facet_vertices(np.flatnonzero((co[:, 1] < 0.01) | (co[:, 0] < 0.01)))
        loads = [(topo.facet_vertices(np.flatnonzero(co[:, 0] > 0.99)), (1000.0, 0.0)),
                 (topo.facet_vertices(vertices_on_line(co, (3, 4))), (1000.0, 1000.0))]
    else:
        raise ValueError(name)
    s = setup.sample
    s.fixed[:] = False
    s.fixed[fixed] = True
    s.rhs[:] = 0
    for v, m in loads:
        s.rhs[v] += m
    return setup, len(c0)


def jittered_case(name: str, levels: int, fraction: float = 0.15, seed: int = 0):
    """``large_case(name, levels)`` with every interior, unconstrained vertex of the last refinement moved by a
    deterministic jitter of at most ``fraction`` x its shortest incident edge: the mesh is then no uniform
    refinement, while ``large_case(name, l)`` for l < levels stay meshes of the same domain.  Returns
    (Sample, n_coarse_vertices); ``levels`` >= 1."""
    setup, n0 = large_case(name, levels)
    s = setup.sample
    co = s.coors.copy()
    conn = np.asarray(s.conn, dtype=np.int64)
    n_prev = len(large_case(name, levels - 1)[0].coors)   # vertices that the last refinement did not add
    e = np.concatenate([conn[:, [0, 1]], conn[:, [1, 2]], conn[:, [2, 0]]])
    e = np.sort(e, axis=1)
    key, cnt = np.unique(e[:, 0] * len(co) + e[:, 1], return_counts=True)
    e0, e1 = key // len(co), key % len(co)
    boundary = np.zeros(len(co), bool)
    boundary[e0[cnt == 1]] = boundary[e1[cnt == 1]] = True
    length = np.linalg.norm(co[e0] - co[e1], axis=1)
    shortest = np.full(len(co), np.inf)
    np.minimum.at(shortest, e0, length)
    np.minimum.at(shortest, e1, length)
    move = np.flatnonzero((np.arange(len(co)) >= n_prev) & ~boundary & ~s.fixed.astype(bool))
    rng = np.random.default_rng(seed)
    ang = rng.uniform(0.0, 2.0 * np.pi, len(move))
    rad = fraction * shortest[move] * rng.uniform(0.0, 1.0, len(move))
    co[move, 0] += rad * np.cos(ang)
    co[move, 1] += rad * np.sin(ang)
    from .solver import Sample
    return Sample(np.ascontiguousarray(co), s.conn, s.cell_region, s.D, s.fixed, s.rhs), n0


def plate_meshes(seed: int, sizes, max_tries: int = 50):
    """One random plate geometry (``PlateGenerator``, seeded) meshed at each of ``sizes``:
    ([(coors, conn) per size], ptags, ltags).  The geometry's corners keep their ids at every size, so
    tag-based conditions mean the same on every mesh."""
    from .plates import GeometryRejected, PlateGenerator
    gen = PlateGenerator(random_seed=seed)
    for _ in range(max_tries):
        g = gen.normalize_geometry(gen.generate_geometry())
        try:
            meshes = []
            for h in sizes:
                ptags, ltags = gen.generate_mesh(g, h)
                meshes.append(gen.mesh)
            return meshes, ptags, ltags
        except GeometryRejected:
            continue
    raise RuntimeError("no plate meshable at every size after %d tries (seed %d)" % (max_tries, seed))


def plate_condition(ptags, ltags) -> Dict:
    """A well-posed condition in the plate's tags: the first exterior edge clamped, a point load at the
    exterior corner after it (FEAnalysis keyword arguments; the default material everywhere)."""
    edge = next(iter(ltags[-1].values()))
    return dict(constraints_edges_tags=[edge], force_vertex_tags_magnitudes=[(ptags[-1][2], (0.0, -1000.0))])
