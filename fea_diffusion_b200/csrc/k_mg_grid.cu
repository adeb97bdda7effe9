// Multigrid hierarchy of a single sample from nested background grids with Galerkin operators
// (fea_batch_set_grid_hierarchy; DESIGN.md section 3.12).  The caller gives no coarse mesh: the coarse levels are
// built here at assemble time, and everything after the build -- transfers, Lanczos estimate, Chebyshev V-cycle,
// coarsest run_pcg, outer flexible CG, load cases -- is the non-nested path of k_mg.cu / k_mg_nonnested.cu.
//
//   grids     : h = sqrt(2 A / NC) (A the summed cell area, in a fixed order: chunks of kSumChunk cells summed in
//               order by one thread each, then the chunk sums by one thread).  Coarse level levels-1 is a grid of
//               spacing 2h, each coarser one doubles it; all share the origin (bounding-box minimum - 1e-10 x its
//               longest side).  Vertex (i, j) = (x0 + i H, y0 + j H) rounded op by op; square (i, j) is split by
//               its diagonal (i, j)-(i+1, j+1).  Level l-1 is then an exact red refinement parent of level l.
//   transfers : the mesh's vertices are located in the finest grid's triangles by mg_locate_points (the rules of
//               section 3.10); grid to grid the weights are 1 and 1/2 of the refinement, in par3 / w3.
//   pruning   : a grid vertex is active when an active vertex of the next finer level gives it a non-zero weight;
//               a triangle is kept when it has an active vertex.  Kept vertices and cells keep grid order
//               (count / scan); kept vertices that are not active are fixed in the level batch.
//   operators : K_(l-1) = P^T K_l P, unscaled, one thread per coarse row: its sorted child list, each child's
//               sorted neighbours, each neighbour's parents, in that order (no floating-point atomics).  The
//               pattern is the sorted union over the same loops.  The level batch's adjacency and block-SELL
//               values come from this block-CSR (api_batch_assemble_csr).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <memory>
#include <vector>

#include "fea_internal.cuh"

namespace fea {

namespace {

constexpr int kT = 256;
constexpr int kSumChunk = 1024;   // cells / vertices one thread folds in order

unsigned blocks(int64_t n) { return (unsigned)((std::max<int64_t>(n, 1) + kT - 1) / kT); }

// chunk t: sum of the cells' |twice area| (shoelace rounded op by op) in order, and the vertices' bounding box
__global__ void k_mgg_chunks(int64_t nc, int64_t nv, int64_t n_chunks, const int32_t* __restrict__ conn,
                             const double* __restrict__ xy, double* __restrict__ part) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_chunks) return;
  double a = 0.0, x0 = INFINITY, x1 = -INFINITY, y0 = INFINITY, y1 = -INFINITY;
  for (int64_t c = t * kSumChunk; c < min(nc, (t + 1) * kSumChunk); ++c) {
    double x[3], y[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      x[k] = xy[2 * (int64_t)conn[3 * c + k]];
      y[k] = xy[2 * (int64_t)conn[3 * c + k] + 1];
    }
    double a2 = 0.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int n = (k + 1) % 3;
      a2 = __dadd_rn(a2, __dsub_rn(__dmul_rn(x[k], y[n]), __dmul_rn(x[n], y[k])));
    }
    a = __dadd_rn(a, fabs(a2));
  }
  for (int64_t v = t * kSumChunk; v < min(nv, (t + 1) * kSumChunk); ++v) {
    x0 = fmin(x0, xy[2 * v]);
    x1 = fmax(x1, xy[2 * v]);
    y0 = fmin(y0, xy[2 * v + 1]);
    y1 = fmax(y1, xy[2 * v + 1]);
  }
  double* p = part + 5 * t;
  p[0] = a;
  p[1] = x0;
  p[2] = x1;
  p[3] = y0;
  p[4] = y1;
}
__global__ void k_mgg_fold(int64_t n_chunks, const double* __restrict__ part, double* __restrict__ out) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  double a = 0.0, x0 = INFINITY, x1 = -INFINITY, y0 = INFINITY, y1 = -INFINITY;
  for (int64_t t = 0; t < n_chunks; ++t) {
    a = __dadd_rn(a, part[5 * t]);
    x0 = fmin(x0, part[5 * t + 1]);
    x1 = fmax(x1, part[5 * t + 2]);
    y0 = fmin(y0, part[5 * t + 3]);
    y1 = fmax(y1, part[5 * t + 4]);
  }
  out[0] = a;
  out[1] = x0;
  out[2] = x1;
  out[3] = y0;
  out[4] = y1;
}

// the full grid of nx x ny squares: vertex (i, j) = j (nx + 1) + i, square s = j nx + i -> triangles 2s, 2s+1
__global__ void k_mgg_grid(int nx, int ny, double x0, double y0, double H, double* __restrict__ xy, int32_t* __restrict__ conn) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nvg = (int64_t)(nx + 1) * (ny + 1);
  if (t < nvg) {
    const int i = (int)(t % (nx + 1)), j = (int)(t / (nx + 1));
    xy[2 * t] = __dadd_rn(x0, __dmul_rn((double)i, H));
    xy[2 * t + 1] = __dadd_rn(y0, __dmul_rn((double)j, H));
  }
  if (t < (int64_t)nx * ny) {
    const int i = (int)(t % nx), j = (int)(t / nx);
    const int v = j * (nx + 1) + i;
    int32_t* c = conn + 6 * t;
    c[0] = v;
    c[1] = v + 1;
    c[2] = v + nx + 2;
    c[3] = v;
    c[4] = v + nx + 2;
    c[5] = v + nx + 1;
  }
}

// act[p] = 1 for every parent p of an active vertex (par3 drops zero weights)
__global__ void k_mgg_mark(int64_t nvf, const int32_t* __restrict__ par3, const uint8_t* __restrict__ fixed_f,
                           uint8_t* __restrict__ act) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nvf || fixed_f[v]) return;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int p = par3[3 * v + k];
    if (p >= 0) act[p] = 1;
  }
}

// triangles with an active vertex are kept, and so are their vertices
__global__ void k_mgg_keep(int64_t ncg, const int32_t* __restrict__ conn, const uint8_t* __restrict__ act,
                           int32_t* __restrict__ cell_kept, int32_t* __restrict__ vtx_kept) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ncg) return;
  const int a = conn[3 * t], b = conn[3 * t + 1], c = conn[3 * t + 2];
  const bool keep = act[a] || act[b] || act[c];
  cell_kept[t] = keep;
  if (keep) vtx_kept[a] = vtx_kept[b] = vtx_kept[c] = 1;
}

// kept vertices in grid order: coordinates, fixed mask (kept but not active), grid index
__global__ void k_mgg_compact_v(int64_t nvg, const int32_t* __restrict__ kept, const int32_t* __restrict__ id,
                                const double2* __restrict__ xyg, const uint8_t* __restrict__ act, double2* __restrict__ xy,
                                uint8_t* __restrict__ fixed, int32_t* __restrict__ grid_of) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nvg || !kept[f]) return;
  const int k = id[f];
  xy[k] = xyg[f];
  fixed[k] = act[f] ? 0 : 1;
  grid_of[k] = (int)f;
}
__global__ void k_mgg_compact_c(int64_t ncg, const int32_t* __restrict__ kept, const int32_t* __restrict__ cid,
                                const int32_t* __restrict__ vid, const int32_t* __restrict__ connf, int32_t* __restrict__ conn,
                                int8_t* __restrict__ creg) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ncg || !kept[t]) return;
  const int k = cid[t];
#pragma unroll
  for (int a = 0; a < 3; ++a) conn[3 * k + a] = vid[connf[3 * t + a]];
  creg[k] = 0;
}

// parents from grid numbering to kept numbering (a parent that is not kept: dropped); cnt[parent] += 1
__global__ void k_mgg_remap(int64_t nvf, int32_t* __restrict__ par3, double* __restrict__ w3, const int32_t* __restrict__ kept,
                            const int32_t* __restrict__ id, int32_t* __restrict__ cnt) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nvf) return;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int p = par3[3 * v + k];
    if (p < 0) continue;
    if (!kept[p]) {
      par3[3 * v + k] = -1;
      w3[3 * v + k] = 0.0;
      continue;
    }
    par3[3 * v + k] = id[p];
    atomicAdd(cnt + id[p], 1);
  }
}

// parents of the kept vertices of a grid (grid_of: their grid index, nx squares a row) in the grid of twice
// the spacing (nxc squares a row): itself (weight 1) at even (i, j), else the two ends of the coarse edge
// (horizontal, vertical or the diagonal) with 1/2 each, ascending
__global__ void k_mgg_grid_parents(int64_t nk, const int32_t* __restrict__ grid_of, int nx, int nxc, int32_t* __restrict__ par3,
                                   double* __restrict__ w3) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nk) return;
  const int f = grid_of[k];
  const int i = f % (nx + 1), j = f / (nx + 1);
  const bool own = !(i & 1) && !(j & 1);
  par3[3 * k] = (j >> 1) * (nxc + 1) + (i >> 1);
  par3[3 * k + 1] = own ? -1 : ((j + 1) >> 1) * (nxc + 1) + ((i + 1) >> 1);
  par3[3 * k + 2] = -1;
  w3[3 * k] = own ? 1.0 : 0.5;
  w3[3 * k + 1] = own ? 0.0 : 0.5;
  w3[3 * k + 2] = 0.0;
}

// Galerkin row of coarse vertex I: count pass (FILL = false: cnt[I] = pattern length, flag[0] |= 1 on overflow,
// flag[1] = longest row) or fill pass (columns and blocks at optr[I]).  Fine rows (fptr, fcol, fval) hold active
// columns only and no row for a fixed vertex, so the fine Dirichlet DOFs drop out.
template <bool FILL>
__global__ void k_mgg_galerkin(int64_t nvc, const uint8_t* __restrict__ fixed_c, const int32_t* __restrict__ child_ptr,
                               const int32_t* __restrict__ child, const double* __restrict__ child_w,
                               const int32_t* __restrict__ fptr, const int32_t* __restrict__ fcol, const d4* __restrict__ fval,
                               const int32_t* __restrict__ par3, const double* __restrict__ w3, int32_t* __restrict__ cnt,
                               int32_t* __restrict__ flag, const int32_t* __restrict__ optr, int32_t* __restrict__ ocol,
                               d4* __restrict__ oval) {
  const int64_t I = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (I >= nvc) return;
  int lst[kMaxAdj];
  int n = 0;
  if (!fixed_c[I]) {
    for (int i = child_ptr[I]; i < child_ptr[I + 1] && n >= 0; ++i) {
      const int a = child[i];
      for (int e = fptr[a]; e < fptr[a + 1] && n >= 0; ++e) {
        const int b = fcol[e];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const int J = par3[3 * (int64_t)b + k];
          if (J < 0 || n < 0) continue;
          int m = 0;
          while (m < n && lst[m] < J) ++m;
          if (m < n && lst[m] == J) continue;
          if (n == kMaxAdj) {
            n = -1;
            continue;
          }
          for (int q = n; q > m; --q) lst[q] = lst[q - 1];
          lst[m] = J;
          ++n;
        }
      }
    }
  }
  if (!FILL) {
    if (n < 0) {
      atomicOr(flag, 1);
      n = 0;
    }
    cnt[I] = n;
    atomicMax(flag + 1, n);
    return;
  }
  if (n <= 0) return;
  double acc[kMaxAdj][4];
  for (int m = 0; m < n; ++m) acc[m][0] = acc[m][1] = acc[m][2] = acc[m][3] = 0.0;
  for (int i = child_ptr[I]; i < child_ptr[I + 1]; ++i) {
    const int a = child[i];
    const double wa = child_w[i];
    for (int e = fptr[a]; e < fptr[a + 1]; ++e) {
      const int b = fcol[e];
      const d4 kb = fval[e];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const int J = par3[3 * (int64_t)b + k];
        if (J < 0) continue;
        int lo = 0, hi = n - 1;   // lst holds J
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (lst[mid] < J) lo = mid + 1; else hi = mid;
        }
        const double c = wa * w3[3 * (int64_t)b + k];
        acc[lo][0] = fma(c, kb.x, acc[lo][0]);
        acc[lo][1] = fma(c, kb.y, acc[lo][1]);
        acc[lo][2] = fma(c, kb.z, acc[lo][2]);
        acc[lo][3] = fma(c, kb.w, acc[lo][3]);
      }
    }
  }
  const int o = optr[I];
  for (int m = 0; m < n; ++m) {
    ocol[o + m] = lst[m];
    d4 v;
    v.x = acc[m][0];
    v.y = acc[m][1];
    v.z = acc[m][2];
    v.w = acc[m][3];
    oval[o + m] = v;
  }
}

// n_cases copies of a block-CSR of nv rows and nnz entries, case k's vertices shifted by k nv
__global__ void k_mgg_replicate_csr(int64_t nv, int64_t nnz, int n_cases, const int32_t* __restrict__ ptr, const int32_t* __restrict__ col,
                                    const d4* __restrict__ val, int32_t* __restrict__ ptr_k, int32_t* __restrict__ col_k,
                                    d4* __restrict__ val_k) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < nnz * n_cases) {
    const int64_t k = t / nnz, e = t - k * nnz;
    col_k[t] = (int32_t)(col[e] + k * nv);
    val_k[t] = val[e];
  }
  if (t <= nv * n_cases) {
    const int64_t k = t / nv, v = t - k * nv;
    ptr_k[t] = (int32_t)(k == n_cases ? n_cases * nnz : ptr[v] + k * nnz);
  }
}

// drop an allocation of b before b is freed
void drop(Batch& b, void* p) {
  if (!p) return;
  cudaFreeAsync(p, b.ctx->stream);
  b.allocs.erase(std::find(b.allocs.begin(), b.allocs.end(), p));
}

struct GridDims {
  int nx = 0, ny = 0;
  double H = 0.0;
  int64_t nv() const { return (int64_t)(nx + 1) * (ny + 1); }
  int64_t nc() const { return 2 * (int64_t)nx * ny; }
};

}  // namespace

int mg_set_grid_hierarchy(fea_ctx* ctx, Batch& b, int levels) {
  (void)ctx;
  std::unique_ptr<Mg> mg(new Mg());
  mg->levels = levels;
  mg->grid = true;
  mg->nonnested = true;   // transfers by weighted parents (par3 / w3)
  mg->lev.resize(levels + 1);
  MgLevel& top = mg->lev[levels];
  top.b = &b;
  top.nv = b.NV;
  top.nc = b.NC;
  b.mg = mg.release();
  return FEA_OK;
}

int mg_grid_assemble(fea_ctx* ctx, Batch& b) {
  Mg& mg = *b.mg;
  cudaStream_t st = ctx->c.stream;
  const int L = mg.levels;
  Scratch scratch(st);
  // mesh size and bounding box
  const int64_t n_chunks = std::max<int64_t>((std::max(b.NC, b.NV) + kSumChunk - 1) / kSumChunk, 1);
  double *part = nullptr, *sums = nullptr;
  CK(ctx, scratch.alloc(&part, 5 * n_chunks));
  CK(ctx, scratch.alloc(&sums, 5));
  k_mgg_chunks<<<blocks(n_chunks), kT, 0, st>>>(b.NC, b.NV, n_chunks, b.conn, b.xy, part);
  k_mgg_fold<<<1, 32, 0, st>>>(n_chunks, part, sums);
  CK(ctx, cudaGetLastError());
  double h_sums[5];
  CK(ctx, cudaMemcpyAsync(h_sums, sums, sizeof h_sums, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  ctx->c.launches += 2;
  if (!(h_sums[0] > 0.0) || !std::isfinite(h_sums[0]))
    return api_fail(ctx, FEA_MESH_ERROR, "the mesh has no area to lay a grid hierarchy over");
  const double h = std::sqrt(h_sums[0] / (double)b.NC);
  const double tol = 1e-10 * std::max(h_sums[2] - h_sums[1], h_sums[4] - h_sums[3]);
  const double x0 = h_sums[1] - tol, x1 = h_sums[2] + tol, y0 = h_sums[3] - tol, y1 = h_sums[4] + tol;
  std::vector<GridDims> g(L);
  {
    const double H0 = (2.0 * h) * (double)(1 << (L - 1));
    auto squares = [H0](double a0, double a1) {
      int64_t k = std::max<int64_t>(1, (int64_t)std::ceil((a1 - a0) / H0));
      while (a0 + (double)k * H0 < a1) ++k;
      return k;
    };
    const int64_t n0x = squares(x0, x1), n0y = squares(y0, y1);
    if (((n0x + 1) << (L - 1)) * ((n0y + 1) << (L - 1)) >= (1LL << 30)) {
      char msg[160];
      snprintf(msg, sizeof msg, "the finest background grid (level %d) would have more than 2^30 vertices", L - 1);
      return api_fail(ctx, FEA_MESH_ERROR, msg);
    }
    for (int l = 0; l < L; ++l) {
      g[l].nx = (int)(n0x << l);
      g[l].ny = (int)(n0y << l);
      g[l].H = H0 / (double)(1 << l);
    }
  }
  // the full grid of level l (scratch)
  auto make_grid = [&](int l, double** xy, int32_t** conn) -> int {
    CK(ctx, scratch.alloc(xy, 2 * g[l].nv()));
    CK(ctx, scratch.alloc(conn, 3 * g[l].nc()));
    k_mgg_grid<<<blocks(std::max(g[l].nv(), g[l].nc() / 2)), kT, 0, st>>>(g[l].nx, g[l].ny, x0, y0, g[l].H, *xy, *conn);
    CK(ctx, cudaGetLastError());
    ctx->c.launches += 1;
    return FEA_OK;
  };
  double* gxy = nullptr;
  int32_t* gconn = nullptr;
  int rc = make_grid(L - 1, &gxy, &gconn);
  if (rc != FEA_OK) return rc;
  {
    const GridDims& f = g[L - 1];
    const double box[4] = {x0, x0 + (double)f.nx * f.H, y0, y0 + (double)f.ny * f.H};
    int32_t* cnt = nullptr;
    CK(ctx, scratch.alloc(&cnt, f.nv() + 1));
    rc = mg_locate_points(ctx, b, L, mg.lev[L], b.NV, b.xy, f.nv(), f.nc(), gconn, gxy, box, cnt);
    if (rc != FEA_OK) return rc;
  }
  // the finest level's unscaled matrix as a block-CSR over its adjacency
  double* mesh_val = nullptr;
  CK(ctx, scratch.alloc(&mesh_val, 4 * b.n_adj));
  CK(ctx, launch_block_csr(b, mesh_val));
  ctx->c.launches += 1;
  int32_t* flag = nullptr;
  CK(ctx, scratch.alloc(&flag, 2));
  for (int l = L - 1; l >= 0; --l) {
    MgLevel& F = mg.lev[l + 1];
    MgLevel& C = mg.lev[l];
    const Batch& fb = *F.b;
    const int64_t nvg = g[l].nv(), ncg = g[l].nc();
    // pruning
    uint8_t* act = nullptr;
    int32_t *vkept = nullptr, *ckept = nullptr, *vid = nullptr, *cid = nullptr, *tmp = nullptr, *cnt = nullptr;
    CK(ctx, scratch.alloc(&act, nvg));
    CK(ctx, scratch.alloc(&vkept, nvg + 1));
    CK(ctx, scratch.alloc(&ckept, ncg + 1));
    CK(ctx, scratch.alloc(&vid, nvg + 1));
    CK(ctx, scratch.alloc(&cid, ncg + 1));
    CK(ctx, scratch.alloc(&tmp, std::max(nvg, ncg) / 4096 + 4));
    CK(ctx, cudaMemsetAsync(act, 0, nvg, st));
    CK(ctx, cudaMemsetAsync(vkept, 0, sizeof(int32_t) * (nvg + 1), st));
    CK(ctx, cudaMemsetAsync(ckept, 0, sizeof(int32_t) * (ncg + 1), st));
    k_mgg_mark<<<blocks(F.nv), kT, 0, st>>>(F.nv, F.par3, fb.fixed, act);
    k_mgg_keep<<<blocks(ncg), kT, 0, st>>>(ncg, gconn, act, ckept, vkept);
    CK(ctx, cudaGetLastError());
    CK(ctx, exclusive_scan_i32(vkept, vid, nvg, tmp, st));
    CK(ctx, exclusive_scan_i32(ckept, cid, ncg, tmp, st));
    int32_t nk = 0, nck = 0;
    CK(ctx, cudaMemcpyAsync(&nk, vid + nvg, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaMemcpyAsync(&nck, cid + ncg, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaStreamSynchronize(st));
    if (nk == 0) return api_fail(ctx, FEA_MESH_ERROR, "the mesh has no active vertex to build a grid hierarchy from");
    // the level batch of the kept triangles
    const int64_t vo[2] = {0, nk}, co[2] = {0, nck};
    const int32_t ro[2] = {0, 1};
    if ((rc = api_batch_begin(ctx, 1, 3, vo, co, ro, &C.hb)) != FEA_OK) return rc;
    Batch& cb = C.hb->b;
    C.b = &cb;
    C.nv = nk;
    C.nc = nck;
    int32_t *grid_of = nullptr, *conn = nullptr;
    int8_t* creg = nullptr;
    CK(ctx, dalloc(cb, &cb.xy, 2 * (int64_t)nk));
    CK(ctx, dalloc(cb, &cb.D, 9));
    CK(ctx, dalloc(cb, &cb.fixed, nk));
    CK(ctx, dalloc(cb, &cb.rhs, 2 * (int64_t)nk));
    CK(ctx, cudaMemsetAsync(cb.D, 0, sizeof(double) * 9, st));
    CK(ctx, cudaMemsetAsync(cb.rhs, 0, sizeof(double) * 2 * nk, st));
    CK(ctx, scratch.alloc(&grid_of, nk));
    CK(ctx, scratch.alloc(&conn, 3 * (int64_t)nck));
    CK(ctx, scratch.alloc(&creg, nck));
    k_mgg_compact_v<<<blocks(nvg), kT, 0, st>>>(nvg, vkept, vid, (const double2*)gxy, act, (double2*)cb.xy, cb.fixed, grid_of);
    k_mgg_compact_c<<<blocks(ncg), kT, 0, st>>>(ncg, ckept, cid, vid, gconn, conn, creg);
    CK(ctx, cudaGetLastError());
    if ((rc = api_batch_finish(ctx, cb, creg, conn)) != FEA_OK) return rc;
    // transfers from this level to the finer one, in kept numbering
    CK(ctx, scratch.alloc(&cnt, (int64_t)nk + 1));
    CK(ctx, cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (nk + 1), st));
    k_mgg_remap<<<blocks(F.nv), kT, 0, st>>>(F.nv, F.par3, F.w3, vkept, vid, cnt);
    CK(ctx, cudaGetLastError());
    if ((rc = mg_child_lists(ctx, b, F, nk, cnt)) != FEA_OK) return rc;
    // Galerkin product
    const int32_t* fptr = l + 1 == L ? b.adj_ptr : F.g_ptr;
    const int32_t* fcol = l + 1 == L ? b.adj : F.g_col;
    const d4* fval = (const d4*)(l + 1 == L ? mesh_val : F.g_val);
    CK(ctx, cudaMemsetAsync(flag, 0, 2 * sizeof(int32_t), st));
    CK(ctx, cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (nk + 1), st));
    k_mgg_galerkin<false><<<blocks(nk), kT, 0, st>>>(nk, cb.fixed, F.child_ptr, F.child, F.child_w, fptr, fcol, fval, F.par3, F.w3,
                                                     cnt, flag, nullptr, nullptr, nullptr);
    CK(ctx, cudaGetLastError());
    CK(ctx, dalloc(cb, &C.g_ptr, (int64_t)nk + 1));
    CK(ctx, exclusive_scan_i32(cnt, C.g_ptr, nk, tmp, st));
    int32_t h_flag[2] = {0, 0}, nnz = 0;
    CK(ctx, cudaMemcpyAsync(h_flag, flag, sizeof h_flag, cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaMemcpyAsync(&nnz, C.g_ptr + nk, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaStreamSynchronize(st));
    if (h_flag[0]) {
      char msg[160];
      snprintf(msg, sizeof msg, "a Galerkin row of grid level %d has more than %d neighbours", l, kMaxAdj - 1);
      return api_fail(ctx, FEA_MESH_ERROR, msg);
    }
    C.g_max_row = h_flag[1];
    CK(ctx, dalloc(cb, &C.g_col, nnz));
    CK(ctx, dalloc(cb, &C.g_val, 4 * (int64_t)nnz));
    k_mgg_galerkin<true><<<blocks(nk), kT, 0, st>>>(nk, cb.fixed, F.child_ptr, F.child, F.child_w, fptr, fcol, fval, F.par3, F.w3,
                                                    nullptr, nullptr, C.g_ptr, C.g_col, (d4*)C.g_val);
    CK(ctx, cudaGetLastError());
    if ((rc = api_batch_assemble_csr(ctx, cb, C.g_ptr, C.g_col, C.g_val, C.g_max_row)) != FEA_OK) return rc;
    ctx->c.launches += 9;
    if (l + 1 < L) {   // the finer grid level's block-CSR has served its product
      drop(*F.b, F.g_ptr);
      drop(*F.b, F.g_col);
      drop(*F.b, F.g_val);
      F.g_ptr = F.g_col = nullptr;
      F.g_val = nullptr;
    }
    if (l == 0) break;
    // the next coarser grid and this level's parents in it
    if ((rc = make_grid(l - 1, &gxy, &gconn)) != FEA_OK) return rc;
    CK(ctx, dalloc(b, &C.par3, 3 * (int64_t)nk));
    CK(ctx, dalloc(b, &C.w3, 3 * (int64_t)nk));
    k_mgg_grid_parents<<<blocks(nk), kT, 0, st>>>(nk, grid_of, g[l].nx, g[l - 1].nx, C.par3, C.w3);
    CK(ctx, cudaGetLastError());
    ctx->c.launches += 1;
  }
  return FEA_OK;
}

int mg_grid_assemble_cases(fea_ctx* ctx, const MgLevel& L0, Batch& kb, int K) {
  cudaStream_t st = ctx->c.stream;
  const int64_t nv = L0.nv;
  int32_t nnz = 0;
  CK(ctx, cudaMemcpyAsync(&nnz, L0.g_ptr + nv, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  Scratch scratch(st);
  int32_t *ptr = nullptr, *col = nullptr;
  double* val = nullptr;
  CK(ctx, scratch.alloc(&ptr, K * nv + 1));
  CK(ctx, scratch.alloc(&col, K * (int64_t)nnz));
  CK(ctx, scratch.alloc(&val, 4 * K * (int64_t)nnz));
  k_mgg_replicate_csr<<<blocks(std::max<int64_t>(K * (int64_t)nnz, K * nv + 1)), kT, 0, st>>>(
      nv, nnz, K, L0.g_ptr, L0.g_col, (const d4*)L0.g_val, ptr, col, (d4*)val);
  CK(ctx, cudaGetLastError());
  ctx->c.launches += 1;
  return api_batch_assemble_csr(ctx, kb, ptr, col, val, L0.g_max_row);
}

}  // namespace fea
