// Multigrid hierarchy of a single sample whose coarser levels are the caller's own meshes of the same domain
// (fea_batch_set_coarse_meshes; DESIGN.md section 3.10).  Only the transfers are new; the V-cycle, the
// smoothers, the coarsest solve and the outer flexible CG are those of k_mg.cu.
//
//   levels    : every coarse mesh is an internal single-sample Batch (fea_batch_create on its slice of the
//               description); at assemble its operator is its own stiffness matrix (rediscretised).
//   location  : the triangles of level l-1 are bucketed into a uniform grid (about one grid cell per
//               triangle) by their bounding boxes grown by the tolerance; one thread per vertex of level l
//               tests the triangles of its grid cell.  Containment is edge-inclusive and rounded op by op
//               (__dmul_rn / __dsub_rn, no FMA contraction); the lowest-index containing triangle wins.  A
//               vertex outside every triangle takes the nearest one within tol = 1e-10 * the longest side of
//               level l-1's bounding box (ties: lowest index), with its barycentric weights clamped to
//               [0, 1] and renormalised; farther out it is a FEA_MESH_ERROR.
//   transfers : up to 3 (parent, weight) pairs per vertex, weights of 0 dropped; restriction gathers over a
//               per-coarse-vertex (fine vertex, weight) list sorted by fine vertex.  No floating-point atomics.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <memory>
#include <vector>

#include "fea_internal.cuh"

namespace fea {

namespace {

constexpr int kT = 256;

struct Grid {
  double x0, y0, inv_hx, inv_hy;
  int nx, ny;
};

__device__ __forceinline__ int bin_of(double v, double v0, double inv_h, int n) {
  const double t = floor(__dmul_rn(__dsub_rn(v, v0), inv_h));
  return t < 0.0 ? 0 : t >= (double)n ? n - 1 : (int)t;
}

// grid cells covered by a triangle's bounding box grown by tol: count (cur == nullptr) or fill
__global__ void k_mgn_bin(int64_t nc, const int32_t* __restrict__ conn, const double2* __restrict__ xy, Grid g, double tol,
                          const int32_t* __restrict__ ptr, int32_t* __restrict__ cnt, int32_t* __restrict__ list) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nc) return;
  const double2 a = xy[conn[3 * t]], b = xy[conn[3 * t + 1]], c = xy[conn[3 * t + 2]];
  const int ix0 = bin_of(__dsub_rn(fmin(a.x, fmin(b.x, c.x)), tol), g.x0, g.inv_hx, g.nx);
  const int ix1 = bin_of(__dadd_rn(fmax(a.x, fmax(b.x, c.x)), tol), g.x0, g.inv_hx, g.nx);
  const int iy0 = bin_of(__dsub_rn(fmin(a.y, fmin(b.y, c.y)), tol), g.y0, g.inv_hy, g.ny);
  const int iy1 = bin_of(__dadd_rn(fmax(a.y, fmax(b.y, c.y)), tol), g.y0, g.inv_hy, g.ny);
  for (int iy = iy0; iy <= iy1; ++iy)
    for (int ix = ix0; ix <= ix1; ++ix) {
      const int cell = iy * g.nx + ix;
      if (!list) atomicAdd(cnt + cell, 1);
      else list[ptr[cell] + atomicAdd(cnt + cell, 1)] = (int)t;
    }
}

// twice the signed area of (a, b, p), rounded op by op
__device__ __forceinline__ double edge_fn(double2 a, double2 b, double2 p) {
  return __dsub_rn(__dmul_rn(__dsub_rn(b.x, a.x), __dsub_rn(p.y, a.y)), __dmul_rn(__dsub_rn(b.y, a.y), __dsub_rn(p.x, a.x)));
}
// squared distance from p to the segment ab
__device__ __forceinline__ double seg_d2(double2 a, double2 b, double2 p) {
  const double abx = __dsub_rn(b.x, a.x), aby = __dsub_rn(b.y, a.y);
  const double apx = __dsub_rn(p.x, a.x), apy = __dsub_rn(p.y, a.y);
  const double ll = __dadd_rn(__dmul_rn(abx, abx), __dmul_rn(aby, aby));
  double t = ll > 0.0 ? __ddiv_rn(__dadd_rn(__dmul_rn(apx, abx), __dmul_rn(apy, aby)), ll) : 0.0;
  t = fmin(fmax(t, 0.0), 1.0);
  const double dx = __dsub_rn(apx, __dmul_rn(t, abx)), dy = __dsub_rn(apy, __dmul_rn(t, aby));
  return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
}

// one thread per vertex of level l: parents and weights in level l-1; cnt[parent] += 1 per kept parent;
// *bad = lowest vertex farther than tol from every triangle
__global__ void k_mgn_locate(int64_t nvf, const double2* __restrict__ xyf, const int32_t* __restrict__ conn,
                             const double2* __restrict__ xyc, Grid g, double tol2, const int32_t* __restrict__ ptr,
                             const int32_t* __restrict__ list, int32_t* __restrict__ par3, double* __restrict__ w3,
                             int32_t* __restrict__ cnt, int32_t* __restrict__ bad) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nvf) return;
  const double2 p = xyf[v];
  const int cell = bin_of(p.y, g.y0, g.inv_hy, g.ny) * g.nx + bin_of(p.x, g.x0, g.inv_hx, g.nx);
  int best_in = INT_MAX, best_near = INT_MAX;
  double best_d2 = INFINITY;
  for (int i = ptr[cell]; i < ptr[cell + 1]; ++i) {
    const int t = list[i];
    const double2 a = xyc[conn[3 * t]], b = xyc[conn[3 * t + 1]], c = xyc[conn[3 * t + 2]];
    const double e0 = edge_fn(a, b, p), e1 = edge_fn(b, c, p), e2 = edge_fn(c, a, p);
    if ((e0 >= 0.0 && e1 >= 0.0 && e2 >= 0.0) || (e0 <= 0.0 && e1 <= 0.0 && e2 <= 0.0)) {
      best_in = min(best_in, t);
    } else if (best_in == INT_MAX) {
      const double d2 = fmin(seg_d2(a, b, p), fmin(seg_d2(b, c, p), seg_d2(c, a, p)));
      if (d2 < best_d2 || (d2 == best_d2 && t < best_near)) {
        best_d2 = d2;
        best_near = t;
      }
    }
  }
  const bool inside = best_in != INT_MAX;
  if (!inside && !(best_d2 <= tol2)) {
    atomicMin(bad, (int)v);
    return;
  }
  const int t = inside ? best_in : best_near;
  const int id[3] = {conn[3 * t], conn[3 * t + 1], conn[3 * t + 2]};
  const double2 a = xyc[id[0]], b = xyc[id[1]], c = xyc[id[2]];
  const double e0 = edge_fn(a, b, p), e1 = edge_fn(b, c, p), e2 = edge_fn(c, a, p);
  const double s = __dadd_rn(__dadd_rn(e0, e1), e2);
  double w[3] = {__ddiv_rn(e1, s), __ddiv_rn(e2, s), __ddiv_rn(e0, s)};   // weights of a, b, c
  if (!inside) {
#pragma unroll
    for (int k = 0; k < 3; ++k) w[k] = fmin(fmax(w[k], 0.0), 1.0);
    const double sw = __dadd_rn(__dadd_rn(w[0], w[1]), w[2]);
#pragma unroll
    for (int k = 0; k < 3; ++k) w[k] = __ddiv_rn(w[k], sw);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const bool keep = w[k] != 0.0;
    par3[3 * v + k] = keep ? id[k] : -1;
    w3[3 * v + k] = keep ? w[k] : 0.0;
    if (keep) atomicAdd(cnt + id[k], 1);
  }
}

__global__ void k_mgn_child_fill(int64_t nvf, const int32_t* __restrict__ par3, const double* __restrict__ w3,
                                 const int32_t* __restrict__ ptr, int32_t* __restrict__ cur, int32_t* __restrict__ child,
                                 double* __restrict__ child_w) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nvf) return;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int p = par3[3 * v + k];
    if (p < 0) continue;
    const int slot = ptr[p] + atomicAdd(cur + p, 1);
    child[slot] = (int)v;
    child_w[slot] = w3[3 * v + k];
  }
}

// insertion sort of each coarse vertex's (fine vertex, weight) list by fine vertex (distinct keys)
__global__ void k_mgn_child_sort(int64_t nvc, const int32_t* __restrict__ ptr, int32_t* __restrict__ child,
                                 double* __restrict__ child_w) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nvc) return;
  const int b = ptr[v], e = ptr[v + 1];
  for (int i = b + 1; i < e; ++i) {
    const int t = child[i];
    const double tw = child_w[i];
    int j = i - 1;
    while (j >= b && child[j] > t) {
      child[j + 1] = child[j];
      child_w[j + 1] = child_w[j];
      --j;
    }
    child[j + 1] = t;
    child_w[j + 1] = tw;
  }
}

unsigned blocks(int64_t n) { return (unsigned)((std::max<int64_t>(n, 1) + kT - 1) / kT); }

}  // namespace

// parents and weights (F.par3, F.w3) of the nvf points xyf of level l in the triangles of level l-1 (nvc vertices
// xyc, ncc triangles connc inside the box [x0, x1] x [y0, y1]); cnt[nvc + 1] (zeroed here) counts each parent's
// kept entries
int mg_locate_points(fea_ctx* ctx, Batch& top, int l, MgLevel& F, int64_t nvf, const double* xyf, int64_t nvc, int64_t ncc,
                     const int32_t* connc, const double* xyc, const double box[4], int32_t* cnt) {
  cudaStream_t st = ctx->c.stream;
  const double x0 = box[0], x1 = box[1], y0 = box[2], y1 = box[3];
  const double W = x1 - x0, H = y1 - y0, tol = 1e-10 * std::max(W, H);
  // about one grid cell per coarse triangle, square cells
  const double hg = std::sqrt(std::max(W * H, 1e-300) / (double)std::max<int64_t>(ncc, 1));
  Grid g;
  g.x0 = x0;
  g.y0 = y0;
  g.nx = W > 0.0 ? (int)std::min<double>(std::ceil(W / hg), 4096.0) : 1;
  g.ny = H > 0.0 ? (int)std::min<double>(std::ceil(H / hg), 4096.0) : 1;
  g.nx = std::max(g.nx, 1);
  g.ny = std::max(g.ny, 1);
  g.inv_hx = W > 0.0 ? g.nx / W : 0.0;
  g.inv_hy = H > 0.0 ? g.ny / H : 0.0;
  const int64_t ncell = (int64_t)g.nx * g.ny;
  Scratch scratch(st);
  int32_t *gcnt = nullptr, *gptr = nullptr, *tmp = nullptr, *bad = nullptr, *glist = nullptr;
  CK(ctx, scratch.alloc(&gcnt, ncell + 1));
  CK(ctx, scratch.alloc(&gptr, ncell + 1));
  CK(ctx, scratch.alloc(&tmp, ncell / 4096 + 4));
  CK(ctx, scratch.alloc(&bad, 1));
  CK(ctx, cudaMemsetAsync(gcnt, 0, sizeof(int32_t) * (ncell + 1), st));
  k_mgn_bin<<<blocks(ncc), kT, 0, st>>>(ncc, connc, (const double2*)xyc, g, tol, nullptr, gcnt, nullptr);
  CK(ctx, cudaGetLastError());
  CK(ctx, exclusive_scan_i32(gcnt, gptr, ncell, tmp, st));
  int32_t total = 0;
  CK(ctx, cudaMemcpyAsync(&total, gptr + ncell, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  CK(ctx, scratch.alloc(&glist, total));
  CK(ctx, cudaMemsetAsync(gcnt, 0, sizeof(int32_t) * (ncell + 1), st));
  k_mgn_bin<<<blocks(ncc), kT, 0, st>>>(ncc, connc, (const double2*)xyc, g, tol, gptr, gcnt, glist);
  CK(ctx, cudaGetLastError());
  CK(ctx, dalloc(top, &F.par3, 3 * nvf));
  CK(ctx, dalloc(top, &F.w3, 3 * nvf));
  CK(ctx, cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (nvc + 1), st));
  const int32_t none = INT_MAX;
  CK(ctx, cudaMemcpyAsync(bad, &none, sizeof(int32_t), cudaMemcpyHostToDevice, st));
  k_mgn_locate<<<blocks(nvf), kT, 0, st>>>(nvf, (const double2*)xyf, connc, (const double2*)xyc, g, tol * tol, gptr, glist,
                                           F.par3, F.w3, cnt, bad);
  CK(ctx, cudaGetLastError());
  int32_t h_bad = INT_MAX;
  CK(ctx, cudaMemcpyAsync(&h_bad, bad, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  ctx->c.launches += 3;
  if (h_bad != INT_MAX) {
    char msg[200];
    snprintf(msg, sizeof msg, "vertex %d of level %d lies outside every triangle of level %d by more than %.3g", h_bad, l,
             l - 1, tol);
    return api_fail(ctx, FEA_MESH_ERROR, msg);
  }
  return FEA_OK;
}

// restriction lists of F's parents in a level of nvc vertices: scan of cnt (entries per parent), fill, sort
int mg_child_lists(fea_ctx* ctx, Batch& top, MgLevel& F, int64_t nvc, int32_t* cnt) {
  cudaStream_t st = ctx->c.stream;
  Scratch scratch(st);
  int32_t* tmp = nullptr;
  CK(ctx, scratch.alloc(&tmp, nvc / 4096 + 4));
  CK(ctx, dalloc(top, &F.child_ptr, nvc + 1));
  CK(ctx, exclusive_scan_i32(cnt, F.child_ptr, nvc, tmp, st));
  int32_t n_child = 0;
  CK(ctx, cudaMemcpyAsync(&n_child, F.child_ptr + nvc, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  CK(ctx, dalloc(top, &F.child, n_child));
  CK(ctx, dalloc(top, &F.child_w, n_child));
  CK(ctx, cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (nvc + 1), st));
  k_mgn_child_fill<<<blocks(F.nv), kT, 0, st>>>(F.nv, F.par3, F.w3, F.child_ptr, cnt, F.child, F.child_w);
  k_mgn_child_sort<<<blocks(nvc), kT, 0, st>>>(nvc, F.child_ptr, F.child, F.child_w);
  CK(ctx, cudaGetLastError());
  ctx->c.launches += 3;
  return FEA_OK;
}

namespace {

// parents of level l's vertices in level l-1 (coarse: C, its host coordinates for the bounding box)
int locate_level(fea_ctx* ctx, Batch& top, int l, MgLevel& F, MgLevel& C, const double* xy_host) {
  double box[4] = {xy_host[0], xy_host[0], xy_host[1], xy_host[1]};
  for (int64_t i = 1; i < C.nv; ++i) {
    box[0] = std::min(box[0], xy_host[2 * i]);
    box[1] = std::max(box[1], xy_host[2 * i]);
    box[2] = std::min(box[2], xy_host[2 * i + 1]);
    box[3] = std::max(box[3], xy_host[2 * i + 1]);
  }
  Scratch scratch(ctx->c.stream);
  int32_t* cnt = nullptr;
  CK(ctx, scratch.alloc(&cnt, C.nv + 1));
  int rc = mg_locate_points(ctx, top, l, F, F.nv, F.b->xy, C.nv, C.nc, C.b->conn, C.b->xy, box, cnt);
  if (rc == FEA_OK) rc = mg_child_lists(ctx, top, F, C.nv, cnt);
  return rc;
}

}  // namespace

int mg_set_coarse_meshes(fea_ctx* ctx, Batch& b, const fea_batch_desc* d) {
  const int n = d->n_samples;
  std::vector<std::unique_ptr<fea_batch, decltype(&api_free_batch)>> owned;
  std::unique_ptr<Mg> mg(new Mg());
  mg->levels = n;
  mg->nonnested = true;
  mg->lev.resize(n + 1);
  for (int s = 0; s < n; ++s) {
    const int64_t v0 = d->vtx_off[s], c0 = d->cell_off[s];
    const int32_t r0 = d->reg_off[s];
    const int64_t nv = d->vtx_off[s + 1] - v0, nc = d->cell_off[s + 1] - c0;
    const int32_t nr = d->reg_off[s + 1] - r0;
    const int32_t* conn = d->conn + 3 * c0;
    for (int64_t i = 0; i < 3 * nc; ++i)
      if (conn[i] < 0 || conn[i] >= nv) {
        char msg[160];
        snprintf(msg, sizeof msg, "coarse mesh %d (level %d): connectivity index out of range", s, s);
        return api_fail(ctx, FEA_MESH_ERROR, msg);
      }
    // one single-sample batch per level; rhs is not read (the restriction writes the coarsest level's)
    const int64_t vo[2] = {0, nv}, co[2] = {0, nc};
    const int32_t ro[2] = {0, nr};
    std::vector<double> zero(2 * std::max<int64_t>(nv, 1), 0.0);
    fea_batch_desc one{1, 3, vo, co, ro, d->xy + 2 * v0, conn, d->cell_region + c0, d->D + 9 * (int64_t)r0, d->fixed + v0,
                       zero.data()};
    fea_batch* hb = nullptr;
    const int rc = fea_batch_create(ctx, &one, &hb);
    if (rc != FEA_OK) return rc;
    owned.emplace_back(hb, api_free_batch);
    MgLevel& L = mg->lev[s];
    L.hb = hb;
    L.b = &hb->b;
    L.nv = nv;
    L.nc = nc;
  }
  MgLevel& top = mg->lev[n];
  top.b = &b;
  top.nv = b.NV;
  top.nc = b.NC;
  for (int l = 1; l <= n; ++l) {
    const int rc = locate_level(ctx, b, l, mg->lev[l], mg->lev[l - 1], d->xy + 2 * d->vtx_off[l - 1]);
    if (rc != FEA_OK) return rc;
  }
  for (auto& o : owned) o.release();   // mg_release frees them from now on
  b.mg = mg.release();
  return FEA_OK;
}

int mg_level_transfer(fea_ctx* ctx, Batch& b, int level, int32_t* indptr, int32_t* indices, double* data) {
  const Mg& mg = *b.mg;
  const MgLevel& F = mg.lev[level];
  const MgLevel& C = mg.lev[level - 1];
  cudaStream_t st = ctx->c.stream;
  std::vector<int32_t> rf(F.nv), rc(C.nv), p3;
  std::vector<double> w3;
  std::vector<int2> p2;
  CK(ctx, cudaMemcpyAsync(rf.data(), F.b->vrank, sizeof(int32_t) * F.nv, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaMemcpyAsync(rc.data(), C.b->vrank, sizeof(int32_t) * C.nv, cudaMemcpyDeviceToHost, st));
  if (mg.nonnested) {
    p3.resize(3 * F.nv);
    w3.resize(3 * F.nv);
    CK(ctx, cudaMemcpyAsync(p3.data(), F.par3, sizeof(int32_t) * 3 * F.nv, cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaMemcpyAsync(w3.data(), F.w3, sizeof(double) * 3 * F.nv, cudaMemcpyDeviceToHost, st));
  } else {
    p2.resize(F.nv);
    CK(ctx, cudaMemcpyAsync(p2.data(), F.par, sizeof(int2) * F.nv, cudaMemcpyDeviceToHost, st));
  }
  CK(ctx, cudaStreamSynchronize(st));
  // active vertices of level l in rank order; each has the same row for both components
  std::vector<int64_t> vert;
  for (int64_t v = 0; v < F.nv; ++v)
    if (rf[v] >= 0) {
      if ((int64_t)vert.size() <= rf[v]) vert.resize(rf[v] + 1, -1);
      vert[rf[v]] = v;
    }
  int64_t nnz = 0;
  if (indptr) indptr[0] = 0;
  for (size_t k = 0; k < vert.size(); ++k) {
    const int64_t v = vert[k];
    std::pair<int32_t, double> e[3];
    int m = 0;
    for (int j = 0; j < 3; ++j) {
      int32_t p = -1;
      double w = 0.0;
      if (mg.nonnested) {
        p = p3[3 * v + j];
        w = w3[3 * v + j];
      } else if (j < 2) {
        const int2 pr = p2[v];
        p = j ? pr.y : pr.x;
        w = pr.y < 0 ? 1.0 : 0.5;
      }
      if (p >= 0 && rc[p] >= 0) e[m++] = {rc[p], w};
    }
    std::sort(e, e + m, [](const std::pair<int32_t, double>& a, const std::pair<int32_t, double>& c) { return a.first < c.first; });
    for (int comp = 0; comp < 2; ++comp) {
      for (int i = 0; i < m; ++i, ++nnz) {
        if (indices) indices[nnz] = 2 * e[i].first + comp;
        if (data) data[nnz] = e[i].second;
      }
      if (indptr) indptr[2 * k + comp + 1] = (int32_t)nnz;
    }
  }
  return FEA_OK;
}

}  // namespace fea
