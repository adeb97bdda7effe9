"""Host-side objects over the C-ABI: samples, packed batches, contexts.

A *sample* is one plate-condition: mesh + Dirichlet vertex mask + material cells + final-step
load.  ``pack`` concatenates samples into the flat arrays ``fea_batch_desc`` expects; ``Context``
owns a ``fea_ctx`` (one GPU, one stream); ``Batch`` wraps the staged life cycle
create -> assemble -> solve -> rasterize -> download.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from . import _capi
from ._capi import BatchDesc, BatchInfo, CoarseInfo, ConditionsDesc, FeaError, MgLevel, SolveStats, ptr


@dataclass
class Sample:
    """Inputs of one plate-condition problem (what FEAnalysis.__init__ derives through sfepy,
    reference datagen/fea_analysis.py:61-164)."""
    coors: np.ndarray        # (n_v, 2) f64
    conn: np.ndarray         # (n_cell, k) i32, as read from the mesh file
    cell_region: np.ndarray  # (n_cell,) i8, -1 = no stiffness
    D: np.ndarray            # (n_reg, 3, 3) f64
    fixed: np.ndarray        # (n_v,) bool / u8
    rhs: np.ndarray          # (n_v, 2) f64 final-step load (N_regions * sum of magnitudes)


class PackedBatch:
    """Concatenated, C-contiguous host arrays + the ctypes descriptor that points at them."""

    def __init__(self, samples: Sequence[Sample], alloc=None):
        """``alloc(shape, dtype)`` may supply page-locked arrays (Context.pinned_empty)."""
        if not samples:
            raise ValueError("empty batch")
        k = samples[0].conn.shape[1]
        if any(s.conn.shape[1] != k for s in samples):
            raise ValueError("all samples of a batch must use the same cell type")
        self.n = len(samples)
        self.k = k
        nv = np.array([len(s.coors) for s in samples], dtype=np.int64)
        nc = np.array([len(s.conn) for s in samples], dtype=np.int64)
        nr = np.array([len(s.D) for s in samples], dtype=np.int64)
        self.vtx_off = np.concatenate([[0], np.cumsum(nv)]).astype(np.int64)
        self.cell_off = np.concatenate([[0], np.cumsum(nc)]).astype(np.int64)
        self.reg_off = np.concatenate([[0], np.cumsum(nr)]).astype(np.int32)
        def cat(parts):
            a = np.concatenate(parts)
            if alloc is None:
                return a
            out = alloc(a.shape, a.dtype)
            out[...] = a
            return out
        self.xy = np.ascontiguousarray(cat([np.asarray(s.coors, dtype=np.float64).reshape(-1, 2) for s in samples]))
        self.conn = np.ascontiguousarray(cat([np.asarray(s.conn, dtype=np.int32) for s in samples]))
        self.cell_region = np.ascontiguousarray(cat([np.asarray(s.cell_region, dtype=np.int8) for s in samples]))
        self.D = np.ascontiguousarray(cat([np.asarray(s.D, dtype=np.float64).reshape(-1, 3, 3) for s in samples]))
        self.fixed = np.ascontiguousarray(cat([np.asarray(s.fixed).astype(np.uint8) for s in samples]))
        self.rhs = np.ascontiguousarray(cat([np.asarray(s.rhs, dtype=np.float64).reshape(-1, 2) for s in samples]))
        self.desc = BatchDesc(
            n_samples=self.n, nodes_per_cell=k,
            vtx_off=ptr(self.vtx_off), cell_off=ptr(self.cell_off), reg_off=ptr(self.reg_off),
            xy=ptr(self.xy), conn=ptr(self.conn), cell_region=ptr(self.cell_region),
            D=ptr(self.D), fixed=ptr(self.fixed), rhs=ptr(self.rhs))

    @property
    def n_vertices(self) -> int:
        return int(self.vtx_off[-1])

    @property
    def n_cells(self) -> int:
        return int(self.cell_off[-1])

    @property
    def h2d_bytes(self) -> int:
        return int(sum(a.nbytes for a in (self.vtx_off, self.cell_off, self.reg_off, self.xy, self.conn,
                                          self.cell_region, self.D, self.fixed, self.rhs)))

    def split_vertices(self, a: np.ndarray) -> List[np.ndarray]:
        return [a[self.vtx_off[s]:self.vtx_off[s + 1]] for s in range(self.n)]


class PackedConditions:
    """Plate-conditions in the reference's own terms -- tags, magnitudes and material coordinate
    lists, the keyword arguments of ``FEAnalysis.__init__`` (reference fea_analysis.py:32-48) -- packed
    into the flat arrays of ``fea_conditions_desc``.  Region selection, Dirichlet mask, material
    cells, D and the load vector are then derived on the device
    (``Context.create_batch_from_conditions``).

    ``meshes``: sequence of (coors (n_v, 2), conn (n_cell, k)); ``samples``: sequence of
    (mesh index, kwargs) with kwargs as produced by ``plates.condition_kwargs``.
    """

    KINDS = ("VertexForce", "EdgeForce", "VertexConstraint", "EdgeConstraint", "MaterialRegion")

    def __init__(self, meshes: Sequence, samples: Sequence, alloc=None):
        if not meshes or not samples:
            raise ValueError("empty batch")
        k = np.asarray(meshes[0][1]).shape[1]
        self.k, self.n, self.n_meshes = k, len(samples), len(meshes)
        A = (lambda shape, dtype: np.empty(shape, dtype)) if alloc is None else alloc

        def cat(parts, dtype, width):
            total = sum(len(p) for p in parts)
            out = A((total, width) if width else (total,), dtype)
            o = 0
            for p in parts:
                out[o:o + len(p)] = p
                o += len(p)
            return out

        mv = np.array([len(m[0]) for m in meshes], dtype=np.int64)
        mc = np.array([len(m[1]) for m in meshes], dtype=np.int64)
        self.mesh_vtx_off = np.concatenate([[0], np.cumsum(mv)]).astype(np.int64)
        self.mesh_cell_off = np.concatenate([[0], np.cumsum(mc)]).astype(np.int64)
        self.xy = cat([np.asarray(m[0], dtype=np.float64).reshape(-1, 2) for m in meshes], np.float64, 2)
        self.conn = cat([np.asarray(m[1], dtype=np.int32).reshape(-1, k) for m in meshes], np.int32, k)
        self.sample_mesh = np.array([int(m) for m, _ in samples], dtype=np.int32)
        vf_t, vf_m, ef_t, ef_m, vc_t, ec_t, mat_en, mat_xy, dflt = [], [], [], [], [], [], [], [], []
        counts = []
        self.materials: List[List] = []
        f64 = np.float64
        for _, kw in samples:      # (kept lean: this loop is the host cost of a batch; numpy converts at the end)
            vf = kw.get("force_vertex_tags_magnitudes") or ()
            ef = kw.get("force_edges_tags_magnitudes") or ()
            vc = kw.get("constraints_vertex_tags") or ()
            ec = kw.get("constraints_edges_tags") or ()
            mats = kw.get("material_properties_to_vertices")
            for t, m in vf:
                vf_t.append(t)
                vf_m.append(m)
            for t, m in ef:
                ef_t.append(t)
                ef_m.append(m)
            vc_t.extend(vc)
            ec_t.extend(ec)
            n_m = 0
            if mats is not None:
                keys = list(mats)
                n_m = len(keys)
                mat_en.extend(keys)
                for pts in mats.values():
                    mat_xy.append(pts if (isinstance(pts, np.ndarray) and pts.dtype == f64 and pts.ndim == 2)
                                  else np.asarray(pts, dtype=f64).reshape(-1, 2))
                self.materials.append(keys)
            else:
                self.materials.append([])
            dflt.append((kw.get("youngs_modulus", 210000), kw.get("poisson_ratio", 0.3)))
            counts.append((len(vf), len(ef), len(vc), len(ec), n_m))
        cnt = np.asarray(counts, dtype=np.int64).reshape(-1, 5)
        n_vf, n_ef, n_vc, n_ec, n_mat = (cnt[:, i] for i in range(5))
        self._counts = cnt
        self._names = None

        def offs(counts):
            return np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)

        self.vforce_off, self.eforce_off, self.vfix_off = offs(n_vf), offs(n_ef), offs(n_vc)
        self.efix_off, self.mat_off = offs(n_ec), offs(n_mat)
        self.vforce_tag = np.asarray(vf_t, dtype=np.int32).reshape(-1)
        self.vforce_mag = np.asarray(vf_m, dtype=np.float64).reshape(-1, 2)
        self.eforce_tag = np.asarray(ef_t, dtype=np.int32).reshape(-1, 2)
        self.eforce_mag = np.asarray(ef_m, dtype=np.float64).reshape(-1, 2)
        self.vfix_tag = np.asarray(vc_t, dtype=np.int32).reshape(-1)
        self.efix_tag = np.asarray(ec_t, dtype=np.int32).reshape(-1, 2)
        self.mat_E_nu = np.asarray(mat_en, dtype=np.float64).reshape(-1, 2)
        self.mat_coord_off = np.concatenate([[0], np.cumsum([len(c) for c in mat_xy])]).astype(np.int64)
        self.mat_coords = cat(mat_xy, np.float64, 2) if mat_xy else np.zeros((0, 2))
        self.default_E_nu = np.asarray(dflt, dtype=np.float64).reshape(-1, 2)
        self.n_regions = cnt.sum(axis=1)
        nv = mv[self.sample_mesh]
        nc = mc[self.sample_mesh]
        self.vtx_off = np.concatenate([[0], np.cumsum(nv)]).astype(np.int64)
        self.cell_off = np.concatenate([[0], np.cumsum(nc)]).astype(np.int64)
        self.desc = ConditionsDesc(
            n_meshes=self.n_meshes, n_samples=self.n, nodes_per_cell=k, reserved=0,
            mesh_vtx_off=ptr(self.mesh_vtx_off), mesh_cell_off=ptr(self.mesh_cell_off), xy=ptr(self.xy), conn=ptr(self.conn),
            sample_mesh=ptr(self.sample_mesh),
            vforce_off=ptr(self.vforce_off), vforce_tag=ptr(self.vforce_tag), vforce_mag=ptr(self.vforce_mag),
            eforce_off=ptr(self.eforce_off), eforce_tag=ptr(self.eforce_tag), eforce_mag=ptr(self.eforce_mag),
            vfix_off=ptr(self.vfix_off), vfix_tag=ptr(self.vfix_tag), efix_off=ptr(self.efix_off), efix_tag=ptr(self.efix_tag),
            mat_off=ptr(self.mat_off), mat_E_nu=ptr(self.mat_E_nu), mat_coord_off=ptr(self.mat_coord_off),
            mat_coords=ptr(self.mat_coords), default_E_nu=ptr(self.default_E_nu))

    @property
    def names(self) -> List[List[str]]:
        """Region names of every sample, in the order of the device's region rows."""
        if self._names is None:
            self._names = [["%s%d" % (kind, i) for kind, c in zip(self.KINDS, row) for i in range(int(c))]
                           for row in self._counts]
        return self._names

    @property
    def n_vertices(self) -> int:
        return int(self.vtx_off[-1])

    @property
    def n_cells(self) -> int:
        return int(self.cell_off[-1])

    @property
    def h2d_bytes(self) -> int:
        return int(sum(getattr(self, f).nbytes for f in (
            "mesh_vtx_off", "mesh_cell_off", "xy", "conn", "sample_mesh", "vforce_off", "vforce_tag", "vforce_mag",
            "eforce_off", "eforce_tag", "eforce_mag", "vfix_off", "vfix_tag", "efix_off", "efix_tag", "mat_off",
            "mat_E_nu", "mat_coord_off", "mat_coords", "default_E_nu")))

    def split_vertices(self, a: np.ndarray) -> List[np.ndarray]:
        return [a[self.vtx_off[s]:self.vtx_off[s + 1]] for s in range(self.n)]

    def use_device_copy(self, arena: "PinnedArena"):
        """Point the descriptor's big arrays (xy, conn, mat_coords) at the device copy of ``arena``
        (``PinnedArena.upload``): the batch is then created with device-to-device copies."""
        for f in ("xy", "conn", "mat_coords"):
            a = getattr(self, f)
            d = arena.device_address(a)
            if d is not None:
                setattr(self.desc, f, d)
        return self

    def sample_conn(self, s: int) -> np.ndarray:
        m = int(self.sample_mesh[s])
        return self.conn[self.mesh_cell_off[m]:self.mesh_cell_off[m + 1]]

    def sample_coors(self, s: int) -> np.ndarray:
        m = int(self.sample_mesh[s])
        return self.xy[self.mesh_vtx_off[m]:self.mesh_vtx_off[m + 1]]


@dataclass
class DeviceSetup:
    """What the device derived from the conditions (fea_batch_get_setup / _get_materials)."""
    fixed: np.ndarray          # (n_vertices,) uint8
    cell_region: np.ndarray    # (n_cells,) int8
    rhs: np.ndarray            # (n_vertices, 2)
    region_count: List[np.ndarray]   # per sample: vertices of every region
    region_flags: List[np.ndarray]   # per sample: (n_regions, n_v) uint8
    D: List[np.ndarray]        # per sample: (n_used, 3, 3)


def pack(samples: Sequence[Sample], alloc=None) -> PackedBatch:
    return PackedBatch(samples, alloc)


@dataclass
class BatchResult:
    u: np.ndarray          # (n_vertices, 2) final-step displacement
    ranges: np.ndarray     # (n, 4): min ux, max ux, min uy, max uy (final step)
    iters: np.ndarray
    relres: np.ndarray
    status: np.ndarray
    images: Optional[np.ndarray] = None  # (n, 2, size, size) uint8
    stats: Optional[dict] = None


@dataclass
class LoadCaseResult:
    """Outputs of ``Batch.solve_load_cases``: per load case, what ``BatchResult`` holds for the batch's sample."""
    u: np.ndarray          # (K, n_vertices, 2)
    ranges: np.ndarray     # (K, 4): min ux, max ux, min uy, max uy
    iters: np.ndarray      # (K,) outer iterations
    relres: np.ndarray     # (K,)
    status: np.ndarray     # (K,)
    stats: dict            # fea_solve_stats of the call (iterations = the largest outer count)


class PinnedArena:
    """A reusable block of page-locked host memory handed out as numpy arrays: staging buffers of a
    pipeline step are carved from it (``empty``) and recycled with ``reset`` -- no page faults, no
    cudaHostAlloc per step.  Falls back to pageable memory when a request does not fit."""

    def __init__(self, ctx: "Context", nbytes: int):
        self.buf = ctx.pinned_empty((int(nbytes),), np.uint8)
        self.off = 0
        self.spilled = 0

    def reset(self):
        self.off = 0

    def empty(self, shape, dtype) -> np.ndarray:
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        o = (self.off + 63) // 64 * 64
        if o + n > self.buf.size:
            self.spilled += 1
            return np.empty(shape, dtype)
        self.off = o + n
        return self.buf[o:o + n].view(dtype).reshape(shape)

    def upload(self, ctx: "Context"):
        """Copy what has been handed out so far into a device buffer of the same size on ``ctx``'s stream
        (fea_device_upload; returns when the copy is done).  ``ctx`` is the calling thread's own context."""
        if getattr(self, "dev", None) is None:
            self.dev = ctx.device_alloc(self.buf.size)
            self._dev_ctx = ctx
        ctx.device_upload(self.dev, self.buf, self.off)
        return self

    def device_address(self, a: np.ndarray):
        """Device address of an array carved from this arena (None if it lives elsewhere or nothing was uploaded)."""
        if getattr(self, "dev", None) is None or a.size == 0:
            return None
        o = a.ctypes.data - self.buf.ctypes.data
        return self.dev + o if 0 <= o and o + a.nbytes <= self.off else None

    def release_device(self):
        if getattr(self, "dev", None) is not None:
            self._dev_ctx.device_free(self.dev)
            self.dev = None


class Context:
    """One fea_ctx: a GPU and a stream.  Not thread-safe; use one per host thread."""

    def __init__(self, device: int = 0, priority: int = 0):
        self.lib = _capi.load_library()
        h = C.c_void_p()
        rc = self.lib.fea_ctx_create_prio(int(device), int(priority), C.byref(h))
        if rc != 0:
            raise FeaError(rc, "fea_ctx_create(device=%d) failed (no CUDA device?)" % device)
        self.h = h
        self.device = device
        self._pinned = []

    def _check(self, rc: int):
        if rc != 0:
            raise FeaError(rc, self.lib.fea_last_error(self.h).decode("utf-8", "replace"))

    def close(self):
        if getattr(self, "h", None):
            for p in self._pinned:
                self.lib.fea_host_free(self.h, p)
            self._pinned = []
            self.lib.fea_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        self._check(self.lib.fea_ctx_synchronize(self.h))

    def event_record(self, slot: int):
        self._check(self.lib.fea_ctx_event_record(self.h, int(slot)))

    def event_elapsed_ms(self, start: int, stop: int) -> float:
        ms = C.c_float()
        self._check(self.lib.fea_ctx_event_elapsed_ms(self.h, int(start), int(stop), C.byref(ms)))
        return float(ms.value)

    def wait_for(self, other: "Context"):
        """Stream-order this context after everything submitted to ``other`` so far."""
        self._check(self.lib.fea_ctx_wait_ctx(self.h, other.h))

    def set_option(self, key: str, value: int):
        """fea_ctx_set_int: "pcg_path" (0 auto / 1 streaming kernels only), "cluster_min", "cluster_halo_cap",
        "row_order", "refine_rounds" (include/fea_b200.h)."""
        self._check(self.lib.fea_ctx_set_int(self.h, key.encode("ascii"), int(value)))

    def kernel_launches(self) -> int:
        n = C.c_int64()
        self._check(self.lib.fea_ctx_kernel_launches(self.h, C.byref(n)))
        return int(n.value)

    def device_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self._check(self.lib.fea_device_alloc(self.h, int(nbytes), C.byref(p)))
        return int(p.value)

    def device_free(self, dev: int):
        self._check(self.lib.fea_device_free(self.h, C.c_void_p(dev)))

    def device_upload(self, dev: int, host: np.ndarray, nbytes: Optional[int] = None):
        """H2D of the first ``nbytes`` of ``host`` into a ``device_alloc`` buffer; synchronised on return."""
        n = host.nbytes if nbytes is None else int(nbytes)
        self._check(self.lib.fea_device_upload(self.h, C.c_void_p(dev), ptr(host), n))

    def pinned_empty(self, shape, dtype) -> np.ndarray:
        """numpy array over page-locked host memory (fea_host_alloc); released by close() -- the array
        must not be used after that; garbage collection alone never frees it under a live array."""
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        p = C.c_void_p()
        self._check(self.lib.fea_host_alloc(self.h, count * dtype.itemsize, C.byref(p)))
        self._pinned.append(p)
        buf = (C.c_char * max(count * dtype.itemsize, 1)).from_address(p.value)
        buf._owner = self      # the array's base keeps the context (and with it the allocation) alive until
        return np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)   # close() is called explicitly

    def rasterize_fields(self, coors: np.ndarray, conn: np.ndarray, fields: np.ndarray, clim: np.ndarray,
                         affine: np.ndarray, size: int, cell_fields: bool = False) -> np.ndarray:
        """(n_fields, size, size) uint8 images of scalar fields of one mesh (fea_rasterize_fields):
        per-vertex (region flags, the constant field of input.png) or per-cell (stress/strain)."""
        coors = np.ascontiguousarray(coors, dtype=np.float64)
        conn = np.ascontiguousarray(conn, dtype=np.int32)
        fields = np.ascontiguousarray(np.atleast_2d(fields), dtype=np.float64)
        clim = np.ascontiguousarray(clim, dtype=np.float64).reshape(len(fields), 2)
        affine = np.ascontiguousarray(affine, dtype=np.float64).reshape(4)
        if fields.shape[1] != (len(conn) if cell_fields else len(coors)):
            raise ValueError("fields must be (n_fields, n_vertices) or (n_fields, n_cells)")
        out = np.empty((len(fields), int(size), int(size)), np.uint8)
        self._check(self.lib.fea_rasterize_fields(self.h, ptr(coors), len(coors), ptr(conn), len(conn),
                                                  conn.shape[1], ptr(fields), len(fields), int(bool(cell_fields)), ptr(clim),
                                                  ptr(affine),
                                                  int(size), ptr(out)))
        return out

    def create_batch(self, packed: PackedBatch) -> "Batch":
        return Batch(self, packed)

    def create_batch_from_conditions(self, packed: "PackedConditions") -> "Batch":
        """fea_batch_create_from_conditions: region selection / Dirichlet mask / material cells / load on
        the device, from tags, magnitudes and coordinate lists."""
        return Batch(self, packed)

    def solve_batch(self, packed: PackedBatch, rtol: float = 1e-10, max_iter: int = 20000,
                    image_size: int = 0, affine: Optional[np.ndarray] = None, value_scale: float = 1.0,
                    out: Optional[BatchResult] = None) -> BatchResult:
        """One-call host-buffer path (fea_solve_batch): H2D, assemble, solve, rasterise, D2H."""
        n, nv = packed.n, packed.n_vertices
        if out is None:
            out = BatchResult(u=np.empty((nv, 2)), ranges=np.empty((n, 4)), iters=np.empty(n, np.int32),
                              relres=np.empty(n), status=np.empty(n, np.int32))
        if image_size > 0:
            affine = np.ascontiguousarray(affine, dtype=np.float64).reshape(n, 4)
            if out.images is None or out.images.shape != (n, 2, image_size, image_size):
                out.images = np.empty((n, 2, image_size, image_size), np.uint8)
        st = SolveStats()
        self._check(self.lib.fea_solve_batch(
            self.h, C.byref(packed.desc), float(rtol), int(max_iter), int(image_size), ptr(affine),
            float(value_scale), ptr(out.u), ptr(out.ranges), ptr(out.iters), ptr(out.relres), ptr(out.status),
            ptr(out.images) if image_size > 0 else None, C.byref(st)))
        out.stats = st.as_dict()
        return out


class Batch:
    """Staged life cycle of one device-resident batch."""

    def __init__(self, ctx: Context, packed: PackedBatch):
        self.ctx, self.packed = ctx, packed
        h = C.c_void_p()
        if isinstance(packed, PackedConditions):
            ctx._check(ctx.lib.fea_batch_create_from_conditions(ctx.h, C.byref(packed.desc), C.byref(h)))
        else:
            ctx._check(ctx.lib.fea_batch_create(ctx.h, C.byref(packed.desc), C.byref(h)))
        self.h = h
        self.image_size = 0

    def destroy(self):
        if getattr(self, "h", None):
            self.ctx.lib.fea_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.destroy()

    def assemble(self):
        self.ctx._check(self.ctx.lib.fea_batch_assemble(self.h))
        return self

    def solve(self, rtol: float = 1e-10, max_iter: int = 20000):
        self.ctx._check(self.ctx.lib.fea_batch_solve(self.h, float(rtol), int(max_iter)))
        return self

    def rasterize(self, size: int, affine: np.ndarray, value_scale: float = 1.0):
        affine = np.ascontiguousarray(affine, dtype=np.float64).reshape(self.packed.n, 4)
        self.ctx._check(self.ctx.lib.fea_batch_rasterize(self.h, int(size), ptr(affine), float(value_scale)))
        self.image_size = size
        return self

    def download(self, images: bool = False, out: Optional[BatchResult] = None) -> BatchResult:
        """``out`` recycles the host arrays of an earlier result (e.g. pinned ones)."""
        n, nv = self.packed.n, self.packed.n_vertices
        r = out if out is not None else BatchResult(u=np.empty((nv, 2)), ranges=np.empty((n, 4)), iters=np.empty(n, np.int32),
                                                    relres=np.empty(n), status=np.empty(n, np.int32))
        self.ctx._check(self.ctx.lib.fea_batch_download(self.h, ptr(r.u), ptr(r.ranges), ptr(r.iters),
                                                        ptr(r.relres), ptr(r.status)))
        if images:
            if r.images is None or r.images.shape != (n, 2, self.image_size, self.image_size):
                r.images = np.empty((n, 2, self.image_size, self.image_size), np.uint8)
            self.ctx._check(self.ctx.lib.fea_batch_download_images(self.h, ptr(r.images)))
        r.stats = self.stats()
        return r

    def rasterize_flags(self, flags_per_sample: Sequence[np.ndarray]) -> List[np.ndarray]:
        """Region images of every sample: ``flags_per_sample[s]`` is (n_regions_s, n_vertices_s)
        bool/uint8; returns one (n_regions_s, size, size) uint8 array per sample."""
        counts = [len(f) for f in flags_per_sample]
        off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        flat = np.ascontiguousarray(np.concatenate([np.asarray(f, dtype=np.uint8).reshape(-1) for f in flags_per_sample]
                                                   or [np.zeros(0, np.uint8)]))
        out = np.empty((int(off[-1]), self.image_size, self.image_size), np.uint8)
        if off[-1]:
            self.ctx._check(self.ctx.lib.fea_batch_rasterize_flags(self.h, ptr(off), ptr(flat), ptr(out)))
        return [out[off[s]:off[s + 1]] for s in range(len(counts))]

    # ---- batches made from conditions -------------------------------------------------------
    def setup(self, flags: bool = True, counts_only: bool = False) -> DeviceSetup:
        """Download what the device set-up derived (parity tests, text files of the dataset)."""
        p = self.packed
        nv, nc = p.n_vertices, p.n_cells
        nreg = p.n_regions
        cnt = np.empty(int(nreg.sum()), np.int32)
        if counts_only:      # the vertex counts of the regions alone (magnitudes.txt): nothing per vertex or cell is read back
            self.ctx._check(self.ctx.lib.fea_batch_get_setup(self.h, None, None, None, ptr(cnt), None))
            ro = np.concatenate([[0], np.cumsum(nreg)])
            return DeviceSetup(fixed=None, cell_region=None, rhs=None, region_count=[cnt[ro[s]:ro[s + 1]] for s in range(p.n)],
                               region_flags=[], D=[])
        fixed, creg, rhs = np.empty(nv, np.uint8), np.empty(nc, np.int8), np.empty((nv, 2))
        per_v = np.diff(p.vtx_off)
        fl = np.empty(int((nreg * per_v).sum()), np.uint8) if flags else None
        self.ctx._check(self.ctx.lib.fea_batch_get_setup(self.h, ptr(fixed), ptr(creg), ptr(rhs), ptr(cnt), ptr(fl)))
        reg_off, n_used = np.empty(p.n + 1, np.int32), np.empty(p.n, np.int32)
        self.ctx._check(self.ctx.lib.fea_batch_get_materials(self.h, ptr(reg_off), ptr(n_used), None))
        D = np.empty((int(reg_off[-1]), 3, 3))
        self.ctx._check(self.ctx.lib.fea_batch_get_materials(self.h, None, None, ptr(D)))
        ro = np.concatenate([[0], np.cumsum(nreg)])
        fo = np.concatenate([[0], np.cumsum(nreg * per_v)])
        return DeviceSetup(
            fixed=fixed, cell_region=creg, rhs=rhs,
            region_count=[cnt[ro[s]:ro[s + 1]] for s in range(p.n)],
            region_flags=[fl[fo[s]:fo[s + 1]].reshape(int(nreg[s]), int(per_v[s])) for s in range(p.n)] if flags else [],
            D=[D[reg_off[s]:reg_off[s] + n_used[s]] for s in range(p.n)])

    def rasterize_regions(self, with_plate_mask: Optional[Sequence[bool]] = None, out: Optional[np.ndarray] = None) -> List[np.ndarray]:
        """Region images of every sample from the device-resident flags; a sample flagged in
        ``with_plate_mask`` gets the plate mask (input.png) as one more image at the end."""
        p = self.packed
        m = np.zeros(p.n, np.uint8) if with_plate_mask is None else np.ascontiguousarray(with_plate_mask, dtype=np.uint8)
        counts = p.n_regions + m
        off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        shape = (int(off[-1]), self.image_size, self.image_size)
        if out is None or out.size < int(np.prod(shape)):
            out = np.empty(shape, np.uint8)
        else:
            out = out.reshape(-1)[:int(np.prod(shape))].reshape(shape)
        self.ctx._check(self.ctx.lib.fea_batch_rasterize_regions(self.h, ptr(m), ptr(out)))
        return [out[off[s]:off[s + 1]] for s in range(p.n)]

    def classify(self):
        """(floating_parts, empty_vertices) per sample: the derived well-posedness check (A-19)."""
        n = self.packed.n
        a, z = np.empty(n, np.int32), np.empty(n, np.int32)
        self.ctx._check(self.ctx.lib.fea_batch_classify(self.h, ptr(a), ptr(z)))
        return a, z

    def stage_outputs(self, with_plate_mask: Optional[Sequence[bool]] = None):
        """Enqueue the region images (+ plate masks) and the classifier into device buffers and mark the batch
        ready for ``fetch_outputs`` -- no synchronisation (fea_batch_stage_outputs)."""
        m = None if with_plate_mask is None else np.ascontiguousarray(with_plate_mask, dtype=np.uint8)
        self.ctx._check(self.ctx.lib.fea_batch_stage_outputs(self.h, ptr(m)))
        self._stage_mask = m
        return self

    def fetch_outputs(self, copy_ctx: Optional["Context"] = None, out: Optional[BatchResult] = None,
                      regions: Optional[np.ndarray] = None, classifier: bool = True):
        """Read a staged batch back on ``copy_ctx``'s stream (another host thread may call this while the
        batch's own context runs the next batch): (BatchResult with images, region images per sample or None,
        (floating_parts, empty_vertices) or None)."""
        p = self.packed
        c = copy_ctx or self.ctx
        n, size = p.n, self.image_size
        if out is None:
            out = BatchResult(u=np.empty((p.n_vertices, 2)), ranges=np.empty((n, 4)), iters=np.empty(n, np.int32),
                              relres=np.empty(n), status=np.empty(n, np.int32), images=np.empty((n, 2, size, size), np.uint8))
        n_img = C.c_int64()
        c._check(c.lib.fea_batch_staged_region_images(self.h, C.byref(n_img)))
        reg = None
        if n_img.value:
            shape = (n_img.value, size, size)
            reg = np.empty(shape, np.uint8) if regions is None or regions.size < int(np.prod(shape)) else \
                regions.reshape(-1)[:int(np.prod(shape))].reshape(shape)
        cls = (np.empty(n, np.int32), np.empty(n, np.int32)) if classifier and hasattr(p, "n_regions") else None
        c._check(c.lib.fea_batch_fetch_outputs(self.h, c.h if copy_ctx is not None else None, ptr(out.u), ptr(out.ranges),
                                               ptr(out.iters), ptr(out.relres), ptr(out.status), ptr(out.images), ptr(reg),
                                               ptr(cls[0]) if cls else None, ptr(cls[1]) if cls else None))
        per = None
        if reg is not None:
            m = self._stage_mask if getattr(self, "_stage_mask", None) is not None else np.zeros(n, np.uint8)
            off = np.concatenate([[0], np.cumsum(p.n_regions + m)]).astype(np.int64)
            per = [reg[off[s]:off[s + 1]] for s in range(n)]
        return out, per, cls

    CELL_FIELDS = {"stress_x": 0, "stress_y": 1, "strain_x": 2, "strain_y": 3}

    def rasterize_cell_components(self, stress_region: int, names: Sequence[str], value_scale: float = 1.0):
        """Images + final-step ranges of stress / strain components of every sample
        (fea_batch_rasterize_cell_components): ({name: (n, size, size) uint8}, {name: (n, 2) f64})."""
        ids = np.array([self.CELL_FIELDS[nm] for nm in names], np.int32)
        n = self.packed.n
        img = np.empty((len(ids), n, self.image_size, self.image_size), np.uint8)
        rng = np.empty((len(ids), n, 2))
        self.ctx._check(self.ctx.lib.fea_batch_rasterize_cell_components(self.h, int(stress_region), len(ids), ptr(ids),
                                                                         float(value_scale), ptr(img), ptr(rng)))
        return {nm: img[i] for i, nm in enumerate(names)}, {nm: rng[i] for i, nm in enumerate(names)}

    def cell_strain_stress(self, stress_region: int = -1):
        """(strain, stress), each (n_cells, 3): final-step cell averages (e11, e22, 2e12), D*strain."""
        nc = self.packed.n_cells
        strain, stress = np.empty((nc, 3)), np.empty((nc, 3))
        self.ctx._check(self.ctx.lib.fea_batch_cell_strain_stress(self.h, int(stress_region), ptr(strain), ptr(stress)))
        return strain, stress

    def info(self) -> dict:
        i = BatchInfo()
        self.ctx._check(self.ctx.lib.fea_batch_get_info(self.h, C.byref(i)))
        return i.as_dict()

    def stats(self) -> dict:
        s = SolveStats()
        self.ctx._check(self.ctx.lib.fea_batch_get_solve_stats(self.h, C.byref(s)))
        return s.as_dict()

    def refine_rounds(self) -> np.ndarray:
        """Extended-precision rounds per sample (> 0: an ill-conditioned system, see fea_b200.h)."""
        r = np.empty(self.packed.n, np.int32)
        self.ctx._check(self.ctx.lib.fea_batch_get_refine_rounds(self.h, ptr(r)))
        return r

    def timed_launches(self):
        """(spmv_ms, update_ms) arrays: launch t opened iteration 32*t of the last solve."""
        a, u = np.zeros(64, np.float32), np.zeros(64, np.float32)
        n = C.c_int32()
        self.ctx._check(self.ctx.lib.fea_batch_get_timed_launches(self.h, 64, ptr(a), ptr(u), C.byref(n)))
        return a[:n.value].copy(), u[:n.value].copy()

    def sample_sizes(self):
        n = self.packed.n
        a, z = np.empty(n, np.int64), np.empty(n, np.int64)
        self.ctx._check(self.ctx.lib.fea_batch_sample_sizes(self.h, ptr(a), ptr(z)))
        return a, z

    def conn(self):
        c = np.empty((self.packed.n_cells, self.packed.k), np.int32)
        f = np.empty(self.packed.n, np.int32)
        self.ctx._check(self.ctx.lib.fea_batch_get_conn(self.h, ptr(c), ptr(f)))
        return c, f

    def element_stiffness(self) -> np.ndarray:
        k = self.packed.k
        ke = np.empty((self.packed.n_cells, 2 * k, 2 * k))
        self.ctx._check(self.ctx.lib.fea_batch_get_element_stiffness(self.h, ptr(ke)))
        return ke

    def csr(self, sample: int, values: bool = True):
        """scipy CSR of one sample's reduced stiffness matrix in sfepy's layout."""
        import scipy.sparse as sp
        a, z = self.sample_sizes()
        n, nnz = int(a[sample]), int(z[sample])
        indptr = np.empty(n + 1, np.int32)
        indices = np.empty(nnz, np.int32)
        data = np.empty(nnz) if values else None
        self.ctx._check(self.ctx.lib.fea_batch_get_csr(self.h, int(sample), ptr(indptr), ptr(indices), ptr(data)))
        if data is None:
            data = np.ones(nnz)
        return sp.csr_matrix((data, indices, indptr), shape=(n, n))

    def spmv(self, sample: int, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.empty_like(x)
        self.ctx._check(self.ctx.lib.fea_batch_spmv(self.h, int(sample), ptr(x), ptr(y)))
        return y

    # ---- multigrid hierarchy of a uniformly refined single-sample batch ------------------------
    def set_refinement(self, levels: int):
        """Declare the only sample a ``levels``-times uniform red refinement (``workload.refine_uniform``
        numbering); assemble then builds the coarse levels and solve runs multigrid-preconditioned CG."""
        self.ctx._check(self.ctx.lib.fea_batch_set_refinement(self.h, int(levels)))
        return self

    def mg_levels(self) -> List[dict]:
        """Per level, coarsest first: sizes, lambda_max of the scaled operator, V-cycle ms of the last solve."""
        n = C.c_int32()
        self.ctx._check(self.ctx.lib.fea_batch_get_mg_levels(self.h, 0, None, C.byref(n)))
        arr = (MgLevel * n.value)()
        self.ctx._check(self.ctx.lib.fea_batch_get_mg_levels(self.h, n.value, arr, C.byref(n)))
        return [a.as_dict() for a in arr]

    def level_csr(self, level: int):
        """scipy CSR of level ``level``'s Galerkin operator, in the layout of ``csr``."""
        import scipy.sparse as sp
        lv = self.mg_levels()[level]
        n, nnz = int(lv["n_active_dofs"]), int(lv["nnz"])
        indptr, indices, data = np.empty(n + 1, np.int32), np.empty(nnz, np.int32), np.empty(nnz)
        self.ctx._check(self.ctx.lib.fea_batch_get_level_csr(self.h, int(level), ptr(indptr), ptr(indices), ptr(data)))
        return sp.csr_matrix((data, indices, indptr), shape=(n, n))

    def set_coarse_meshes(self, packed: PackedBatch):
        """Declare coarser meshes of the same domain, ``pack([Sample, ...])`` coarsest first (1..8; their rhs is
        not read): assemble then builds a non-nested hierarchy (point location, linear interpolation,
        rediscretised coarse operators) and solve runs multigrid-preconditioned CG."""
        self.ctx._check(self.ctx.lib.fea_batch_set_coarse_meshes(self.h, C.byref(packed.desc)))
        return self

    def set_grid_hierarchy(self, levels: int):
        """Declare ``levels`` (1..8) coarse levels built from the mesh alone: assemble lays nested background
        grids over it (finest spacing twice the mean mesh size), prunes them to the mesh's reach and forms
        Galerkin operators; solve and solve_load_cases then run multigrid-preconditioned CG."""
        self.ctx._check(self.ctx.lib.fea_batch_set_grid_hierarchy(self.h, int(levels)))
        return self

    def level_transfer(self, level: int):
        """scipy CSR of P_level (level-1 -> level) over active DOFs, in the numbering of ``csr``."""
        import scipy.sparse as sp
        lv = self.mg_levels()
        n, m = int(lv[level]["n_active_dofs"]), int(lv[level - 1]["n_active_dofs"])
        indptr = np.empty(n + 1, np.int32)
        self.ctx._check(self.ctx.lib.fea_batch_get_level_transfer(self.h, int(level), ptr(indptr), None, None))
        nnz = int(indptr[-1])
        indices, data = np.empty(nnz, np.int32), np.empty(nnz)
        self.ctx._check(self.ctx.lib.fea_batch_get_level_transfer(self.h, int(level), None, ptr(indices), ptr(data)))
        return sp.csr_matrix((data, indices, indptr), shape=(n, m))

    def solve_load_cases(self, loads: np.ndarray, rtol: float = 1e-10, max_iter: int = 20000) -> LoadCaseResult:
        """Solve K = len(loads) load cases (1..8) of the batch's one sample together with its multigrid hierarchy.
        ``loads`` (K, n_vertices, 2) float64: full-DOF loads like ``Sample.rhs`` (values at fixed DOFs are not
        read).  Case k's outputs equal, bit for bit, those of ``solve`` on a batch whose rhs is loads[k]; the
        batch's own results (``download``) do not change."""
        nv = self.packed.n_vertices
        if not isinstance(loads, np.ndarray) or loads.dtype != np.float64:
            raise TypeError("loads must be a float64 numpy array")
        if loads.ndim != 3 or loads.shape[1:] != (nv, 2):
            raise ValueError("loads must have shape (K, %d, 2), not %s" % (nv, loads.shape))
        loads = np.ascontiguousarray(loads)
        k = loads.shape[0]
        r = LoadCaseResult(u=np.empty((k, nv, 2)), ranges=np.empty((k, 4)), iters=np.empty(k, np.int32),
                           relres=np.empty(k), status=np.empty(k, np.int32), stats={})
        st = SolveStats()
        self.ctx._check(self.ctx.lib.fea_batch_solve_load_cases(
            self.h, int(k), ptr(loads), float(rtol), int(max_iter), ptr(r.u), ptr(r.ranges), ptr(r.iters),
            ptr(r.relres), ptr(r.status), C.byref(st)))
        r.stats = st.as_dict()
        return r

    # ---- outputs of every case of the last solve_load_cases, from the displacements kept on the device ----------
    def load_case_info(self):
        """(K, status (K,) int32, image size) of the fields the last successful ``solve_load_cases`` kept; the image
        size is that of the camera the last ``load_case_images`` kept, 0 before one.  FeaError (BAD_STATE) before
        any such call (fea_batch_load_case_info)."""
        k, size, status = C.c_int32(), C.c_int32(), np.empty(8, np.int32)   # K <= 8
        self.ctx._check(self.ctx.lib.fea_batch_load_case_info(self.h, C.byref(k), ptr(status), C.byref(size)))
        return k.value, status[:k.value].copy(), size.value

    def load_case_images(self, size: int, affine: np.ndarray, value_scale: float = 1.0) -> np.ndarray:
        """Displacement images of every case of the last ``solve_load_cases``: (K, 2, size, size) uint8, case k bit
        for bit those ``rasterize`` + ``download(images=True)`` give a batch solved with loads[k].  ``affine`` holds
        the 4 camera values of the batch's one sample.  The camera is kept for ``load_case_cell_components``."""
        if isinstance(size, bool) or not isinstance(size, (int, np.integer)) or not 1 <= size <= 8192:
            raise ValueError("size must be an integer in 1..8192, not %r" % (size,))
        affine = np.ascontiguousarray(affine, dtype=np.float64)
        if affine.size != 4:
            raise ValueError("affine must hold the 4 camera values of the batch's one sample, not %d" % affine.size)
        k = self.load_case_info()[0]
        img = np.empty((k, 2, int(size), int(size)), np.uint8)
        self.ctx._check(self.ctx.lib.fea_batch_load_case_images(self.h, int(size), ptr(affine.reshape(4)),
                                                                float(value_scale), ptr(img)))
        return img

    def load_case_strain_stress(self, stress_region: int = -1):
        """(strain, stress), each (K, n_cells, 3): ``cell_strain_stress(stress_region)`` of every case of the last
        ``solve_load_cases``, bit for bit."""
        k = self.load_case_info()[0]
        nc = self.packed.n_cells
        strain, stress = np.empty((k, nc, 3)), np.empty((k, nc, 3))
        self.ctx._check(self.ctx.lib.fea_batch_load_case_strain_stress(self.h, int(stress_region), ptr(strain), ptr(stress)))
        return strain, stress

    def load_case_cell_components(self, stress_region: int, names: Sequence[str], value_scale: float = 1.0):
        """``rasterize_cell_components`` of every case of the last ``solve_load_cases``, bit for bit, with the camera of
        the last ``load_case_images``: ({name: (K, size, size) uint8}, {name: (K, 2) f64})."""
        names = list(names)
        if not 1 <= len(names) <= 4 or any(nm not in self.CELL_FIELDS for nm in names):
            raise ValueError("names must be 1..4 of %s, not %r" % (sorted(self.CELL_FIELDS), names))
        k, _, size = self.load_case_info()
        if not size:
            raise FeaError(4, "load_case_cell_components before load_case_images")
        ids = np.array([self.CELL_FIELDS[nm] for nm in names], np.int32)
        img = np.empty((len(ids), k, size, size), np.uint8)
        rng = np.empty((len(ids), k, 2))
        self.ctx._check(self.ctx.lib.fea_batch_load_case_cell_components(self.h, int(stress_region), len(ids), ptr(ids),
                                                                         float(value_scale), ptr(img), ptr(rng)))
        return {nm: img[i] for i, nm in enumerate(names)}, {nm: rng[i] for i, nm in enumerate(names)}

    COARSE_SOLVERS = {"cg": 0, "direct": 1}

    def set_coarse_solver(self, name: str):
        """Choose the coarsest-level solver of the declared hierarchy before ``assemble``: "cg" (block-Jacobi CG to rtol
        1e-4, the default) or "direct" (a dense inverse of level 0, factorised on the device at assemble time)."""
        if not isinstance(name, str) or name not in self.COARSE_SOLVERS:
            raise ValueError("coarse solver must be one of %s, not %r" % (sorted(self.COARSE_SOLVERS), name))
        self.ctx._check(self.ctx.lib.fea_batch_set_coarse_solver(self.h, self.COARSE_SOLVERS[name]))
        return self

    def coarse_info(self) -> dict:
        """solver (0 cg, 1 direct), n, factor_ms, min_pivot and bytes of the assembled coarsest-level solver."""
        i = CoarseInfo()
        self.ctx._check(self.ctx.lib.fea_batch_get_coarse_info(self.h, C.byref(i)))
        return i.as_dict()

    def coarse_solve(self, r: np.ndarray) -> np.ndarray:
        """x = level 0's solver applied to r, a float64 vector over level 0's active DOFs (unscaled, numbered as
        ``level_csr(0)``)."""
        if not isinstance(r, np.ndarray) or r.dtype != np.float64:
            raise TypeError("r must be a float64 numpy array")
        if r.ndim != 1:
            raise ValueError("r must be one vector over level 0's active DOFs, not of shape %s" % (r.shape,))
        n = int(self.mg_levels()[0]["n_active_dofs"])
        if r.shape[0] != n:
            raise ValueError("r must have level 0's %d active DOFs, not %d" % (n, r.shape[0]))
        r = np.ascontiguousarray(r)
        x = np.empty_like(r)
        self.ctx._check(self.ctx.lib.fea_batch_coarse_solve(self.h, ptr(r), ptr(x)))
        return x

    def mg_apply(self, r: np.ndarray) -> np.ndarray:
        """z = M r: one V-cycle on an active-DOF vector of the finest level (unscaled, as ``spmv``)."""
        r = np.ascontiguousarray(r, dtype=np.float64)
        z = np.empty_like(r)
        self.ctx._check(self.ctx.lib.fea_batch_mg_apply(self.h, ptr(r), ptr(z)))
        return z
